// GPU inflate of gzip input (ingest, SURVEY §8(f) next-1: replaces flate2's MultiGzDecoder).
//
// k_inflate_warp inflates block-gzip (BGZF-style) members, which carry their own compressed size ("BC" extra field)
// and are therefore independent streams of at most 64 KiB: one WARP per member, thousands of members per launch,
// table-driven.  All 32 lanes run the same decode (same bit buffer, same tables: no divergence, no broadcasts); the
// lanes differ only where a warp helps: the compressed input arrives through a 512-byte shared-memory ring that the
// lanes top up with coalesced 128-byte loads ahead of the bit reader, Huffman decode is one shared-memory lookup per
// symbol (9-bit table for literal/length codes, 8-bit for distances, built by all lanes from the canonical code;
// longer codes fall back to the bit-by-bit canonical decode), a match is copied by all lanes at once (period `dist`
// when it overlaps itself), and the CRC-32 is computed after the decode, each lane over 1/32 of the output, the
// partial CRCs combined with x^(8n) mod P multiplications.  Each member's CRC-32 and ISIZE (RFC 1952 trailer) are
// checked, as flate2 does; the first bad member is reported.
//
// The k_gz_* kernels further down decode ONE long deflate stream (what `gzip` writes) from speculative block starts,
// with the same warp decoder's tables and symbol loop.
#include "vfb_internal.cuh"

namespace vfb {

#define INF_MAXBITS 15
#define INF_MAXL 288

struct InfTables {
    unsigned short lbase[29], lext[29], dbase[30], dext[30];
    unsigned char order[19];
    uint32_t crc[256];
};

struct InflateArgs {
    const uint8_t *z;            // compressed members, back to back as read from the file
    const vfb_member *members;   // per member: offset/size in z, offset in out, ISIZE
    uint32_t n_members;
    uint8_t *out;
    uint32_t *first_bad;         // atomicMin of the first member that failed
};

#define INFW_WARPS 4
#define INFW_LBITS 9
#define INFW_DBITS 8

struct InfWarp {
    uint32_t ltab[1 << INFW_LBITS];   // nbits | kind << 4 | value << 8 | extra << 24 ; 0 = long / unused code
    uint32_t dtab[1 << INFW_DBITS];   // nbits | extra << 4 | base << 8
    uint16_t lcount[16], dcount[16];  // canonical code: symbols per length
    uint16_t lsym[INF_MAXL], dsym[32];
    uint8_t lens[32 + INF_MAXL + 32];   // code lengths being read (staged 32 bytes up while the code-length code is in use)
    uint32_t ring[128 + 4];           // 4 lines of 32 compressed words; ring[128] mirrors ring[0] (the symbol loop reads
                                      // word pairs without wrapping the second index)
};

struct InfShared {
    InfTables T;
    uint32_t x2n[32];                 // x^(2^n) mod P (reflected CRC-32 polynomial)
    InfWarp w[INFW_WARPS];
};

__device__ __forceinline__ uint32_t crc_multmodp(uint32_t a, uint32_t b)
{
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1u) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}

// x^(n * 2^k) mod P
__device__ uint32_t crc_x2nmodp(const uint32_t *x2n, uint32_t n, uint32_t k)
{
    uint32_t p = 1u << 31;
    while (n) {
        if (n & 1u) p = crc_multmodp(x2n[k & 31], p);
        n >>= 1;
        ++k;
    }
    return p;
}

struct WBits {
    uint64_t buf;
    int cnt;
    uint32_t rw;          // next word (relative to `words`) to enter the bit buffer
    uint32_t next_line;   // next 32-word line to load into the ring
    const uint32_t *words;
    uint32_t nwords;
};

__device__ __forceinline__ void wb_refill(WBits &b, InfWarp *W, int lane)
{
    if (b.cnt > 32) return;
    // (two lines ahead of the word that enters next: the ring's four lines then still hold the line before it, which
    // the symbol loop — it works from a bit position, not from this buffer — may have to read again)
    while (b.next_line <= (b.rw >> 5) + 2) {
        const uint32_t w = b.next_line * 32u + (uint32_t)lane;
        const uint32_t v = w < b.nwords ? __ldg(b.words + w) : 0u;
        W->ring[w & 127u] = v;
        if ((w & 127u) == 0u) W->ring[128] = v;
        ++b.next_line;
        __syncwarp();
    }
    b.buf |= (uint64_t)W->ring[b.rw & 127u] << b.cnt;
    b.cnt += 32;
    ++b.rw;
}

// Start reading at byte `bytepos` (relative to `words`).
__device__ __forceinline__ void wb_seek(WBits &b, InfWarp *W, int lane, uint32_t bytepos)
{
    __syncwarp();
    b.rw = bytepos >> 2;
    b.next_line = b.rw >> 5;
    b.buf = 0;
    b.cnt = 0;
    wb_refill(b, W, lane);
    const int skip = (int)(bytepos & 3u) * 8;
    b.buf >>= skip;
    b.cnt -= skip;
}

__device__ __forceinline__ uint32_t wb_bits(WBits &b, InfWarp *W, int lane, int n)   // n <= 16
{
    wb_refill(b, W, lane);
    const uint32_t v = (uint32_t)b.buf & ((1u << n) - 1u);
    b.buf >>= n;
    b.cnt -= n;
    return v;
}

// bytes consumed so far, rounded up to whole bytes
__device__ __forceinline__ uint32_t wb_bytepos(const WBits &b) { return b.rw * 4u - (uint32_t)(b.cnt >> 3); }

// bit-by-bit canonical decode from the low bits of `bits` (codes are MSB first); returns the
// symbol and its length, or -1
__device__ __forceinline__ int canon_decode(uint32_t bits, const uint16_t *count, const uint16_t *symbol, int maxlen, int *len_out)
{
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= maxlen; ++len) {
        code |= (int)(bits & 1u);
        bits >>= 1;
        const int c = count[len];
        if (code - c < first) {
            *len_out = len;
            return symbol[index + (code - first)];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

// canonical code from code lengths (one lane); <0 over-subscribed, >0 incomplete, 0 complete
__device__ int canon_construct(uint16_t *count, uint16_t *symbol, const uint8_t *length, int n)
{
    uint16_t offs[INF_MAXBITS + 1];
    for (int len = 0; len <= INF_MAXBITS; ++len) count[len] = 0;
    for (int s = 0; s < n; ++s) count[length[s]]++;
    if (count[0] == n) return 0;
    int left = 1;
    for (int len = 1; len <= INF_MAXBITS; ++len) {
        left <<= 1;
        left -= count[len];
        if (left < 0) return left;
    }
    offs[1] = 0;
    for (int len = 1; len < INF_MAXBITS; ++len) offs[len + 1] = offs[len] + count[len];
    for (int s = 0; s < n; ++s)
        if (length[s] != 0) symbol[offs[length[s]]++] = (uint16_t)s;
    return left;
}

__device__ __forceinline__ uint32_t lit_entry(const InfTables *T, int sym, int nbits)
{
    if (sym < 256) return (uint32_t)nbits | ((uint32_t)sym << 8);
    if (sym == 256) return (uint32_t)nbits | (2u << 4);
    if (sym > 285) return (uint32_t)nbits | (3u << 4);                         // invalid length symbol
    return (uint32_t)nbits | (1u << 4) | ((uint32_t)T->lbase[sym - 257] << 8) | ((uint32_t)T->lext[sym - 257] << 24);
}

__device__ __forceinline__ uint32_t dist_entry(const InfTables *T, int sym, int nbits)
{
    if (sym > 29) return (uint32_t)nbits | (15u << 4);                         // invalid distance symbol (extra 15 never occurs)
    return (uint32_t)nbits | ((uint32_t)T->dext[sym] << 4) | ((uint32_t)T->dbase[sym] << 8);
}

// lengths of the literal/length code in W->lens[0..nlen), of the distance code behind them
__device__ int infw_build(const InfTables *T, InfWarp *W, int nlen, int ndist, int lane, bool fixed)
{
    int e1 = 0, e2 = 0;
    if (lane == 0) {
        // an incomplete code is accepted only as a single code of length 1 (zlib's inflate_table)
        e1 = canon_construct(W->lcount, W->lsym, W->lens, nlen);
        if (!(e1 < 0 || (e1 > 0 && !(nlen - W->lcount[0] == 1 && W->lcount[1] == 1)))) e1 = 0; else e1 = 1;
        e2 = canon_construct(W->dcount, W->dsym, W->lens + nlen, ndist);
        if (!(e2 < 0 || (e2 > 0 && !(ndist - W->dcount[0] == 1 && W->dcount[1] == 1)))) e2 = 0; else e2 = 1;
        if (fixed) e1 = e2 = 0;            // the fixed distance code leaves two codes unused (RFC 1951 3.2.6)
    }
    e1 = __shfl_sync(0xffffffffu, e1, 0);
    e2 = __shfl_sync(0xffffffffu, e2, 0);
    if (e1) return -11;
    if (e2) return -12;
    __syncwarp();
    for (int e = lane; e < (1 << INFW_LBITS); e += 32) {
        int len = 0;
        const int sym = canon_decode((uint32_t)e, W->lcount, W->lsym, INFW_LBITS, &len);
        W->ltab[e] = sym < 0 ? 0u : lit_entry(T, sym, len);
    }
    for (int e = lane; e < (1 << INFW_DBITS); e += 32) {
        int len = 0;
        const int sym = canon_decode((uint32_t)e, W->dcount, W->dsym, INFW_DBITS, &len);
        W->dtab[e] = sym < 0 ? 0u : dist_entry(T, sym, len);
    }
    __syncwarp();
    // Literal runs: where the index bits behind a literal's code hold one or two more complete literal
    // codes, the entry decodes them all at once -- bytes in bits 8-15 / 16-23 / 24-31, (count - 1) in bits
    // 6-7, total code length in bits 0-3.  Read text is mostly literals with 2-3 bit codes (the bases), so
    // most look-ups then yield three bytes.  Every lane first derives its entries from the single-symbol
    // table, then all write.
    uint32_t fused[(1 << INFW_LBITS) / 32];
#pragma unroll
    for (int k = 0; k < (1 << INFW_LBITS) / 32; ++k) {
        const uint32_t e = (uint32_t)lane + 32u * (uint32_t)k;
        uint32_t a = W->ltab[e];
        if (a != 0 && ((a >> 4) & 3u) == 0) {
            uint32_t used = a & 15u, cnt = 1, bytes = (a >> 8) & 0xFFu;
            while (cnt < 3 && used < INFW_LBITS) {
                const uint32_t nx = W->ltab[e >> used];             // the bits above `used`, zero-extended
                const uint32_t nb = nx & 15u;
                if (nx == 0 || ((nx >> 4) & 3u) != 0 || used + nb > INFW_LBITS) break;   // not a literal fully inside the index
                bytes |= ((nx >> 8) & 0xFFu) << (8 * cnt);
                used += nb;
                ++cnt;
            }
            a = used | ((cnt - 1) << 6) | (bytes << 8);
        }
        fused[k] = a;
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < (1 << INFW_LBITS) / 32; ++k) W->ltab[lane + 32 * k] = fused[k];
    __syncwarp();
    return 0;
}

__device__ int inflate_member_warp(const InfShared *S, InfWarp *W, const uint8_t *zin, uint32_t zlen, uint8_t *out,
                                   uint32_t isize, int lane)
{
    const InfTables *T = &S->T;
    if (zlen < 18 || zin[0] != 0x1f || zin[1] != 0x8b || zin[2] != 8) return -1;
    const uint32_t flg = zin[3];
    uint32_t p = 10;
    if (flg & 4) { if (p + 2 > zlen) return -1; p += 2 + (zin[p] | (zin[p + 1] << 8)); }
    if (flg & 8) { while (p < zlen && zin[p]) ++p; ++p; }
    if (flg & 16) { while (p < zlen && zin[p]) ++p; ++p; }
    if (flg & 2) p += 2;
    if (p + 8 > zlen) return -1;
    const uint8_t *tr = zin + zlen - 8;
    const uint32_t want_crc = tr[0] | (tr[1] << 8) | (tr[2] << 16) | ((uint32_t)tr[3] << 24);
    const uint32_t want_len = tr[4] | (tr[5] << 8) | (tr[6] << 16) | ((uint32_t)tr[7] << 24);
    if (want_len != isize) return -2;

    WBits b;
    const uintptr_t a0 = reinterpret_cast<uintptr_t>(zin + p);
    b.words = reinterpret_cast<const uint32_t *>(a0 & ~(uintptr_t)3);
    const uint32_t lead = (uint32_t)(a0 & 3u);
    const uint32_t data_len = zlen - 8 - p;                  // deflate stream bytes
    b.nwords = (lead + data_len + 8 + 3) >> 2;               // (the trailer may be looked at, never beyond)
    wb_seek(b, W, lane, lead);
    uint32_t n_out = 0;
    int last;
    do {
        last = (int)wb_bits(b, W, lane, 1);
        const uint32_t type = wb_bits(b, W, lane, 2);
        if (type == 0) {
            const int drop = b.cnt & 7;
            b.buf >>= drop; b.cnt -= drop;
            const uint32_t len = wb_bits(b, W, lane, 16), nlen = wb_bits(b, W, lane, 16);
            if ((len ^ 0xFFFFu) != nlen) return -3;
            if (n_out + len > isize) return -4;
            const uint32_t src = wb_bytepos(b);              // byte aligned here
            if (src + len > lead + data_len) return -19;
            const uint8_t *sp = reinterpret_cast<const uint8_t *>(b.words) + src;
            for (uint32_t i = lane; i < len; i += 32) out[n_out + i] = __ldg(sp + i);
            n_out += len;
            wb_seek(b, W, lane, src + len);
        } else if (type == 1 || type == 2) {
            int nl, nd;
            if (type == 1) {
                nl = 288; nd = 30;
                for (int s = lane; s < 288; s += 32) W->lens[s] = (uint8_t)(s < 144 ? 8 : (s < 256 ? 9 : (s < 280 ? 7 : 8)));
                if (lane < 30) W->lens[288 + lane] = 5;
                __syncwarp();
            } else {
                nl = (int)wb_bits(b, W, lane, 5) + 257;
                nd = (int)wb_bits(b, W, lane, 5) + 1;
                const int ncode = (int)wb_bits(b, W, lane, 4) + 4;
                if (nl > 286 || nd > 30) return -5;
                __syncwarp();
                if (lane < 19) W->lens[lane] = 0;
                __syncwarp();
                for (int idx = 0; idx < ncode; ++idx) {
                    const uint32_t v = wb_bits(b, W, lane, 3);
                    if (lane == 0) W->lens[T->order[idx]] = (uint8_t)v;
                }
                __syncwarp();
                int e0 = 0;
                if (lane == 0) e0 = canon_construct(W->lcount, W->lsym, W->lens, 19);
                e0 = __shfl_sync(0xffffffffu, e0, 0);
                if (e0 != 0) return -6;                          // must be complete
                __syncwarp();
                int idx = 0;
                while (idx < nl + nd) {
                    wb_refill(b, W, lane);
                    int cl = 0;
                    const int sym = canon_decode((uint32_t)b.buf, W->lcount, W->lsym, 7, &cl);
                    if (sym < 0) return -7;
                    b.buf >>= cl; b.cnt -= cl;
                    if (sym < 16) {
                        if (lane == 0) W->lens[32 + idx] = (uint8_t)sym;      // (kept clear of the 19 code-length lengths)
                        ++idx;
                    } else {
                        int len = 0, rep;
                        if (sym == 16) {
                            if (idx == 0) return -8;
                            __syncwarp();
                            len = W->lens[32 + idx - 1];
                            rep = 3 + (int)wb_bits(b, W, lane, 2);
                        } else if (sym == 17) rep = 3 + (int)wb_bits(b, W, lane, 3);
                        else rep = 11 + (int)wb_bits(b, W, lane, 7);
                        if (idx + rep > nl + nd) return -9;
                        if (lane < rep) W->lens[32 + idx + lane] = (uint8_t)len;
                        if (lane + 32 < rep) W->lens[32 + idx + lane + 32] = (uint8_t)len;
                        if (lane + 64 < rep) W->lens[32 + idx + lane + 64] = (uint8_t)len;
                        if (lane + 96 < rep) W->lens[32 + idx + lane + 96] = (uint8_t)len;
                        if (lane + 128 < rep) W->lens[32 + idx + lane + 128] = (uint8_t)len;
                        idx += rep;
                    }
                    __syncwarp();
                }
                // move the lengths down to lens[0..nl+nd)
                uint8_t t[10];
#pragma unroll
                for (int k = 0; k < 10; ++k) t[k] = lane + 32 * k < nl + nd ? W->lens[32 + lane + 32 * k] : (uint8_t)0;
                __syncwarp();
#pragma unroll
                for (int k = 0; k < 10; ++k) if (lane + 32 * k < nl + nd) W->lens[lane + 32 * k] = t[k];
                __syncwarp();
                if (W->lens[256] == 0) return -10;
            }
            const int brc = infw_build(T, W, nl, nd, lane, type == 1);
            if (brc) return brc;
            // ---- the symbol loop.  The bit buffer of the header code gives way to a bit POSITION `bp` (relative to
            // b.words): a symbol starts by fetching the 32 bits at bp — two ring words and a funnel shift, no buffer
            // to shift and count down — and a literal/length code with its extra bits (<= 20 bits) or a distance
            // code with its extra bits (<= 28 bits) is taken out of that one window.  `thr` is the position from which
            // the ring needs its next line (lines up to two ahead of the reader are kept loaded, the line behind it stays).
            {
                uint32_t bp = b.rw * 32u - (uint32_t)b.cnt;
                uint32_t thr = (b.next_line - 2u) << 10;
                const uint32_t *ring = W->ring;
                const uint32_t lane_sh = 8u + 8u * (uint32_t)(lane < 2 ? lane : 2);
                uint8_t *out_lane = out + lane;
                // One way out of the loop (`status`: 1 = end of block, anything else an error code): early returns from
                // inside it cost several reconvergence instructions per symbol.
                int status = 0;
                do {
                    while (bp >= thr) {                            // (rarely taken: once per 128 bytes of input)
                        const uint32_t w = b.next_line * 32u + (uint32_t)lane;
                        const uint32_t v = w < b.nwords ? __ldg(b.words + w) : 0u;
                        W->ring[w & 127u] = v;
                        if ((w & 127u) == 0u) W->ring[128] = v;
                        ++b.next_line;
                        thr += 1024u;
                        __syncwarp();
                    }
                    const uint32_t i0 = (bp >> 5) & 127u;
                    const uint32_t win = __funnelshift_r(ring[i0], ring[i0 + 1], bp);
                    uint32_t e = W->ltab[win & ((1u << INFW_LBITS) - 1u)];
                    if (e == 0) {
                        int cl = 0;
                        const int sym = canon_decode(win, W->lcount, W->lsym, INF_MAXBITS, &cl);
                        e = sym < 0 ? (1u | (3u << 4)) : lit_entry(T, sym, cl);      // no such code: an invalid entry
                    }
                    const uint32_t nb = e & 15u, kind = e & 0x30u;
                    bp += nb;
                    if (kind == 0) {
                        // one to three literals per look-up: bytes in bits 8.., (count - 1) in bits 6-7
                        const uint32_t c1 = (e >> 6) & 3u;
                        if (n_out + c1 < isize) {
                            if ((uint32_t)lane <= c1) out_lane[n_out] = (uint8_t)(e >> lane_sh);
                            n_out += c1 + 1u;
                        } else {
                            status = -14;
                        }
                    } else if (kind == 0x10u) {
                        const uint32_t xb = e >> 24;
                        const uint32_t len = ((e >> 8) & 0xFFFFu) + ((win >> nb) & ~(0xFFFFFFFFu << xb));
                        bp += xb;
                        const uint32_t j0 = (bp >> 5) & 127u;
                        const uint32_t win2 = __funnelshift_r(ring[j0], ring[j0 + 1], bp);
                        uint32_t d = W->dtab[win2 & ((1u << INFW_DBITS) - 1u)];
                        if (d == 0) {
                            int cl = 0;
                            const int ds = canon_decode(win2, W->dcount, W->dsym, INF_MAXBITS, &cl);
                            d = ds < 0 ? (1u | (15u << 4)) : dist_entry(T, ds, cl);  // no such code: an invalid entry
                        }
                        const uint32_t db = d & 15u, dx = (d >> 4) & 15u;
                        // (dx = 15 marks an invalid distance symbol: its 15 "extra bits" only yield a distance that is checked
                        // like any other and then rejected by the flag)
                        const uint32_t dist = (d >> 8) + ((win2 >> db) & ~(0xFFFFFFFFu << dx));
                        bp += db + dx;
                        if (dx != 15u && dist <= n_out && n_out + len <= isize) {
                            __syncwarp();                             // earlier stores of all lanes are visible
                            const uint8_t *from = out_lane + (n_out - dist);
                            if (dist >= len) {
                                // (most matches in read text are a few bases long: one predicated load / store)
                                if (len <= 32) {
                                    if ((uint32_t)lane < len) out_lane[n_out] = __ldcg(from);
                                } else {
                                    for (uint32_t i = 0; i + lane < len; i += 32) out_lane[n_out + i] = __ldcg(from + i);
                                }
                            } else {
                                for (uint32_t i = lane; i < len; i += 32) out[n_out + i] = __ldcg(out + (n_out - dist) + i % dist);
                            }
                            n_out += len;
                        } else {
                            status = dx == 15u ? -16 : (dist > n_out ? -17 : -18);
                        }
                    } else {
                        status = kind == 0x20u ? 1 : (nb == 1u && e == (1u | (3u << 4)) ? -13 : -15);
                    }
                } while (status == 0);
                if (status != 1) return status;
                // back to the bit buffer for the next block header / the trailer check
                b.rw = bp >> 5;
                b.buf = (uint64_t)(W->ring[b.rw & 127u] >> (bp & 31u));
                b.cnt = 32 - (int)(bp & 31u);
                ++b.rw;
            }
        } else {
            return -20;
        }
    } while (!last);
    if (n_out != isize) return -21;
    // the gzip trailer follows the deflate stream at the next byte boundary (RFC 1952)
    if (wb_bytepos(b) != lead + data_len) return -19;
    // CRC-32 of the output: one slice per lane, then combine
    __syncwarp();
    const uint32_t chunk = (isize + 31u) / 32u;
    const uint32_t lo = min(isize, (uint32_t)lane * chunk), hi = min(isize, lo + chunk);
    uint32_t crc = 0xFFFFFFFFu;
    {
        // bytes up to the first 16-byte boundary, then 16 bytes per load (two loads in flight), then the rest
        uint32_t i = lo;
        while (i < hi && ((reinterpret_cast<uintptr_t>(out) + i) & 15u)) { crc = T->crc[(crc ^ __ldcg(out + i)) & 0xFFu] ^ (crc >> 8); ++i; }
        auto word = [&](uint32_t w) {
#pragma unroll
            for (int k = 0; k < 4; ++k) { crc = T->crc[(crc ^ w) & 0xFFu] ^ (crc >> 8); w >>= 8; }
        };
        for (; i + 32 <= hi; i += 32) {
            const uint4 a = __ldcg(reinterpret_cast<const uint4 *>(out + i)), c = __ldcg(reinterpret_cast<const uint4 *>(out + i + 16));
            word(a.x); word(a.y); word(a.z); word(a.w); word(c.x); word(c.y); word(c.z); word(c.w);
        }
        for (; i < hi; ++i) crc = T->crc[(crc ^ __ldcg(out + i)) & 0xFFu] ^ (crc >> 8);
    }
    crc ^= 0xFFFFFFFFu;
    uint32_t total = __shfl_sync(0xffffffffu, crc, 0);
    if (chunk) {
        const uint32_t q_full = crc_x2nmodp(S->x2n, chunk, 3);
        for (int l = 1; l < 32; ++l) {
            const uint32_t c_l = __shfl_sync(0xffffffffu, crc, l);
            const uint32_t l_lo = min(isize, (uint32_t)l * chunk), l_len = min(isize, l_lo + chunk) - l_lo;
            if (l_len == 0) break;
            const uint32_t q = l_len == chunk ? q_full : crc_x2nmodp(S->x2n, l_len, 3);
            total = crc_multmodp(q, total) ^ c_l;
        }
    }
    if (total != want_crc) return -22;
    return 0;
}

// Occupancy: a member is one long serial chain (a launch of 2048 members takes 4.9 ms, one of 4096 members 5.5 ms), so
// throughput is members in flight per SM: the tables are sized (9-bit literal/length look-up, 20 KB per block) and the
// registers capped (40) for 11 blocks = 44 members per SM; at 6500 members per launch 55.6 GB/s of text (32 per SM: 48.3).
__global__ void __launch_bounds__(INFW_WARPS * 32, 11)
k_inflate_warp(const __grid_constant__ InflateArgs a)
{
    __shared__ InfShared S;
    if (threadIdx.x == 0) {
        const unsigned short lb[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
        const unsigned short le[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
        const unsigned short db[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
        const unsigned short de[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
        const unsigned char od[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        for (int i = 0; i < 29; ++i) { S.T.lbase[i] = lb[i]; S.T.lext[i] = le[i]; }
        for (int i = 0; i < 30; ++i) { S.T.dbase[i] = db[i]; S.T.dext[i] = de[i]; }
        for (int i = 0; i < 19; ++i) S.T.order[i] = od[i];
        uint32_t p = 1u << 30;                     // x^1
        S.x2n[0] = p;
        for (int n = 1; n < 32; ++n) S.x2n[n] = p = crc_multmodp(p, p);
    }
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        uint32_t c = (uint32_t)i;
        for (int k = 0; k < 8; ++k) c = (c & 1u) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
        S.T.crc[i] = c;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t warps_total = gridDim.x * INFW_WARPS;
    for (uint32_t i = blockIdx.x * INFW_WARPS + warp; i < a.n_members; i += warps_total) {
        const vfb_member m = a.members[i];
        int rc = 0;
        if (m.isize || m.z_len) rc = inflate_member_warp(&S, &S.w[warp], a.z + m.z_off, m.z_len, a.out + m.out_off, m.isize, lane);
        if (rc != 0 && lane == 0) atomicMin(a.first_bad, i);
        __syncwarp();
    }
}

// =====================================================================================
// Single-stream gzip on the device (SURVEY §8(f) next-1; replaces flate2's MultiGzDecoder, /root/reference/src/lib.rs:233,
// for input that is ONE long deflate stream — what `gzip` writes).  A deflate stream has no index, so:
//   k_gz_search   every bit offset of the compressed segment is tried as the start of a dynamic-Huffman block (block
//                 type, field ranges, a complete code-length code, a valid run-length stream, complete literal/length
//                 and distance codes): the offsets that pass are CANDIDATE block starts;
//   k_gz_decode   one warp per candidate decodes from there — the symbol loop of k_inflate_warp writing 16-bit
//                 symbols behind a 32 KiB window of place holders (256 + p = "byte p of the window I cannot see":
//                 matches copy symbols, so unknown bytes propagate) — until a block ends exactly on a later candidate
//                 (or the stream's final block ends);
//   k_gz_chain    one block follows the landings from the segment's known start: the chunks it visits are exactly the
//                 serial decode (a candidate nobody lands on — a false positive — is simply never visited), computes
//                 every visited chunk's incoming window from its predecessor's and the chunks' places in the text;
//   k_gz_resolve  turns the visited chunks' symbols into bytes (place holders through the chunk's window), counts
//                 newlines per 64 KiB piece;  k_gz_crc  CRC-32 of 16 KiB pieces (the host combines them).
// Correctness does not depend on the search: only chunks reached from a true block start are used.
#define GZ_WIN 32768u
#define GZ_NONE 0xFFFFFFFFu

__device__ __forceinline__ uint32_t gz_peek(const uint32_t *z32, uint32_t n_words, uint32_t bit, int n)   // n <= 25
{
    const uint32_t w = bit >> 5;
    const uint32_t a = w < n_words ? __ldg(z32 + w) : 0u, b = w + 1 < n_words ? __ldg(z32 + w + 1) : 0u;
    return __funnelshift_r(a, b, bit) & ((1u << n) - 1u);
}

// Pass 1: one thread per 32-bit word tries its 32 bit offsets against the cheap part of the test — block type, field
// ranges, and a COMPLETE code-length code (Kraft sum over the 3-bit lengths through a 512-entry table of three fields
// at a time) — and lists the few offsets that pass (about 0.2 % of all).  Pass 2 (one thread per listed offset) decodes
// the two code-length sequences and checks what zlib checks.
__global__ void __launch_bounds__(256)
k_gz_search1(const uint32_t *__restrict__ z32, uint32_t n_words, uint32_t lo_bit, uint32_t hi_bit, uint32_t *list,
             uint32_t *n_list, uint32_t list_cap)
{
    __shared__ uint8_t kraft3[512];            // sum of 128 >> v over three 3-bit fields (v = 0 counts nothing)
    for (int i = threadIdx.x; i < 512; i += blockDim.x) {
        uint32_t k = 0;
        for (int f = 0; f < 3; ++f) { const uint32_t v = (i >> (3 * f)) & 7u; if (v) k += 128u >> v; }
        kraft3[i] = (uint8_t)k;
    }
    __syncthreads();
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t w = (lo_bit >> 5) + blockIdx.x * blockDim.x + threadIdx.x; w * 32u < hi_bit && w < n_words; w += stride) {
        const uint32_t w0 = __ldg(z32 + w), w1 = w + 1 < n_words ? __ldg(z32 + w + 1) : 0u, w2 = w + 2 < n_words ? __ldg(z32 + w + 2) : 0u,
                       w3 = w + 3 < n_words ? __ldg(z32 + w + 3) : 0u;
#pragma unroll 4
        for (uint32_t o = 0; o < 32; ++o) {
            const uint32_t x0 = __funnelshift_r(w0, w1, o);
            if ((x0 & 7u) != 4u) continue;                    // BFINAL = 0, BTYPE = 2 (dynamic)
            const uint32_t hlit = (x0 >> 3) & 31u, hdist = (x0 >> 8) & 31u, ncode = ((x0 >> 13) & 15u) + 4u;
            if (hlit > 29u || hdist > 29u) continue;
            const uint32_t p = w * 32u + o;
            if (p < lo_bit || p >= hi_bit) continue;
            const uint32_t x1 = __funnelshift_r(w1, w2, o), x2 = __funnelshift_r(w2, w3, o);
            // the 3-bit lengths: bits 17 .. 17 + 3 * ncode of the window
            unsigned long long f = ((unsigned long long)(x0 >> 17)) | ((unsigned long long)x1 << 15) | ((unsigned long long)x2 << 47);
            f &= (1ull << (3u * ncode)) - 1ull;               // ncode <= 19: at most 57 bits
            uint32_t k = 0;
#pragma unroll
            for (int g = 0; g < 7; ++g) k += kraft3[(uint32_t)(f >> (9 * g)) & 511u];
            if (k != 128u) continue;
            const uint32_t at = atomicAdd(n_list, 1u);
            if (at < list_cap) list[at] = p;
        }
    }
}

__global__ void __launch_bounds__(128)
k_gz_search2(const uint32_t *__restrict__ z32, uint32_t n_words, const uint32_t *__restrict__ list, const uint32_t *n_list,
             uint32_t list_cap, uint32_t *cand, uint32_t *n_cand, uint32_t cand_cap)
{
    uint32_t n = *n_list;
    if (n > list_cap) n = list_cap;
    const uint32_t total_bits = n_words * 32u;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
        const uint32_t p = list[t];
        const uint32_t hdr = gz_peek(z32, n_words, p, 17);
        const uint32_t hlit = (hdr >> 3) & 31u, hdist = (hdr >> 8) & 31u, ncode = ((hdr >> 13) & 15u) + 4u;
        const unsigned char order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        uint32_t bit = p + 17u;
        uint8_t cl[19];
#pragma unroll
        for (int i = 0; i < 19; ++i) cl[i] = 0;
        for (uint32_t i = 0; i < ncode; ++i) {
            cl[order[i]] = (uint8_t)gz_peek(z32, n_words, bit, 3);
            bit += 3;
        }
        // canonical code over the 19 symbols
        uint8_t count[8], symbol[19], offs[8];
#pragma unroll
        for (int l = 0; l < 8; ++l) count[l] = 0;
        for (int sy = 0; sy < 19; ++sy) count[cl[sy]]++;
        offs[1] = 0;
        for (int l = 1; l < 7; ++l) offs[l + 1] = (uint8_t)(offs[l] + count[l]);
        for (int sy = 0; sy < 19; ++sy)
            if (cl[sy]) symbol[offs[cl[sy]]++] = (uint8_t)sy;
        // the literal/length and distance code lengths
        const uint32_t nl = hlit + 257u, nall = nl + hdist + 1u;
        uint32_t lk = 0, dk = 0, dcodes = 0, dmax = 0;        // Kraft sums in units of 2^-15, distance code count / longest
        uint32_t idx = 0, prev = 0, len256 = 0;
        bool ok = true;
        while (idx < nall && ok) {
            const uint32_t bits = gz_peek(z32, n_words, bit, 7);
            int code = 0, first = 0, index = 0, sym = -1, used = 0;
            for (int l = 1; l <= 7; ++l) {
                code |= (int)((bits >> (l - 1)) & 1u);
                const int c = count[l];
                if (code - c < first) { sym = symbol[index + (code - first)]; used = l; break; }
                index += c; first += c; first <<= 1; code <<= 1;
            }
            if (sym < 0) { ok = false; break; }
            bit += (uint32_t)used;
            uint32_t rep = 1, val = (uint32_t)sym;
            if (sym == 16) {
                if (idx == 0) { ok = false; break; }
                val = prev; rep = 3u + gz_peek(z32, n_words, bit, 2); bit += 2;
            } else if (sym == 17) { val = 0; rep = 3u + gz_peek(z32, n_words, bit, 3); bit += 3; }
            else if (sym == 18) { val = 0; rep = 11u + gz_peek(z32, n_words, bit, 7); bit += 7; }
            if (idx + rep > nall) { ok = false; break; }
            for (uint32_t r = 0; r < rep; ++r, ++idx) {
                if (val) {
                    if (idx < nl) lk += 32768u >> val;
                    else { dk += 32768u >> val; ++dcodes; if (val > dmax) dmax = val; }
                }
                if (idx == 256u) len256 = val;
            }
            prev = val;
        }
        if (!ok || bit > total_bits) continue;
        if (len256 == 0 || lk != 32768u) continue;
        if (!(dk == 32768u || dcodes == 0 || (dcodes == 1 && dmax == 1))) continue;
        const uint32_t k = atomicAdd(n_cand, 1u);
        if (k < cand_cap) cand[k] = p;
    }
}

struct __align__(16) GzChunkRes {
    uint32_t n_sym;      // symbols decoded (without the window prefix)
    uint32_t land;       // chunk on whose start the decode ended, GZ_NONE if none
    uint32_t end_bit;    // bit position where the decode stopped
    uint32_t flags;      // 1 = the stream's final block ended here, 2 = the decode failed / ran out of room
    uint32_t start_bit;  // where the chunk starts (0xFFFFFFFF in the records of landing spots that are not decoded)
    uint32_t pad[3];
};

static_assert(sizeof(GzChunkRes) == VFB_GZ_RES_BYTES, "GzChunkRes layout");

struct GzDecodeArgs {
    const uint32_t *z32;         // compressed segment, word aligned
    uint32_t n_words;
    const uint32_t *starts;      // sorted bit positions of the chunk starts; starts[0] is the segment's true start
    uint32_t n_chunks;
    uint32_t n_decode;           // the first n_decode chunks are decoded (the others are landing spots only)
    uint16_t *out16;             // n_decode regions of (GZ_WIN + cap) symbols
    uint32_t cap;                // output symbols per chunk
    uint32_t max_span_bits;      // compressed bits a chunk may consume
    GzChunkRes *res;
};

// first index j in [lo, n) with starts[j] >= pos
__device__ __forceinline__ uint32_t gz_lower_bound(const uint32_t *starts, uint32_t lo, uint32_t n, uint32_t pos)
{
    uint32_t hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(starts + mid) < pos) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ int gz_chunk_warp(const InfShared *S, InfWarp *W, const GzDecodeArgs &a, uint32_t self, int lane, GzChunkRes *res)
{
    const InfTables *T = &S->T;
    const uint32_t start_bit = a.starts[self];
    uint16_t *region = a.out16 + (size_t)self * (GZ_WIN + (size_t)a.cap);
    uint16_t *o16 = region + GZ_WIN;
    // the window this chunk cannot see: place holders
    {
        uint4 *r4 = reinterpret_cast<uint4 *>(region);
        for (uint32_t k = lane; k < GZ_WIN / 8; k += 32) {
            const uint32_t v = 256u + 8u * k;
            r4[k] = make_uint4(v | ((v + 1) << 16), (v + 2) | ((v + 3) << 16), (v + 4) | ((v + 5) << 16), (v + 6) | ((v + 7) << 16));
        }
    }
    WBits b;
    b.words = a.z32;
    b.nwords = a.n_words;
    wb_seek(b, W, lane, start_bit >> 3);
    { const int skip = (int)(start_bit & 7u); b.buf >>= skip; b.cnt -= skip; }
    const uint32_t cap = a.cap;
    uint32_t n_out = 0;
    const uint32_t next_start = self + 1 < a.n_chunks ? a.starts[self + 1] : GZ_NONE;
    res->land = GZ_NONE;
    res->flags = 0;
    for (;;) {
        const int last = (int)wb_bits(b, W, lane, 1);
        const uint32_t type = wb_bits(b, W, lane, 2);
        if (type == 0) {
            const int drop = b.cnt & 7;
            b.buf >>= drop; b.cnt -= drop;
            const uint32_t len = wb_bits(b, W, lane, 16), nlen = wb_bits(b, W, lane, 16);
            if ((len ^ 0xFFFFu) != nlen) return -3;
            if (n_out + len > cap) return -4;
            const uint32_t src = wb_bytepos(b);              // byte aligned here
            if ((uint64_t)src + len > (uint64_t)a.n_words * 4u) return -19;
            const uint8_t *sp = reinterpret_cast<const uint8_t *>(b.words) + src;
            for (uint32_t i = lane; i < len; i += 32) o16[n_out + i] = (uint16_t)__ldg(sp + i);
            n_out += len;
            wb_seek(b, W, lane, src + len);
        } else if (type == 1 || type == 2) {
            int nl, nd;
            if (type == 1) {
                nl = 288; nd = 30;
                for (int s = lane; s < 288; s += 32) W->lens[s] = (uint8_t)(s < 144 ? 8 : (s < 256 ? 9 : (s < 280 ? 7 : 8)));
                if (lane < 30) W->lens[288 + lane] = 5;
                __syncwarp();
            } else {
                nl = (int)wb_bits(b, W, lane, 5) + 257;
                nd = (int)wb_bits(b, W, lane, 5) + 1;
                const int ncode = (int)wb_bits(b, W, lane, 4) + 4;
                if (nl > 286 || nd > 30) return -5;
                __syncwarp();
                if (lane < 19) W->lens[lane] = 0;
                __syncwarp();
                for (int idx = 0; idx < ncode; ++idx) {
                    const uint32_t v = wb_bits(b, W, lane, 3);
                    if (lane == 0) W->lens[T->order[idx]] = (uint8_t)v;
                }
                __syncwarp();
                int e0 = 0;
                if (lane == 0) e0 = canon_construct(W->lcount, W->lsym, W->lens, 19);
                e0 = __shfl_sync(0xffffffffu, e0, 0);
                if (e0 != 0) return -6;
                __syncwarp();
                int idx = 0;
                while (idx < nl + nd) {
                    wb_refill(b, W, lane);
                    int cl = 0;
                    const int sym = canon_decode((uint32_t)b.buf, W->lcount, W->lsym, 7, &cl);
                    if (sym < 0) return -7;
                    b.buf >>= cl; b.cnt -= cl;
                    if (sym < 16) {
                        if (lane == 0) W->lens[32 + idx] = (uint8_t)sym;
                        ++idx;
                    } else {
                        int len = 0, rep;
                        if (sym == 16) {
                            if (idx == 0) return -8;
                            __syncwarp();
                            len = W->lens[32 + idx - 1];
                            rep = 3 + (int)wb_bits(b, W, lane, 2);
                        } else if (sym == 17) rep = 3 + (int)wb_bits(b, W, lane, 3);
                        else rep = 11 + (int)wb_bits(b, W, lane, 7);
                        if (idx + rep > nl + nd) return -9;
                        if (lane < rep) W->lens[32 + idx + lane] = (uint8_t)len;
                        if (lane + 32 < rep) W->lens[32 + idx + lane + 32] = (uint8_t)len;
                        if (lane + 64 < rep) W->lens[32 + idx + lane + 64] = (uint8_t)len;
                        if (lane + 96 < rep) W->lens[32 + idx + lane + 96] = (uint8_t)len;
                        if (lane + 128 < rep) W->lens[32 + idx + lane + 128] = (uint8_t)len;
                        idx += rep;
                    }
                    __syncwarp();
                }
                uint8_t t[10];
#pragma unroll
                for (int k = 0; k < 10; ++k) t[k] = lane + 32 * k < nl + nd ? W->lens[32 + lane + 32 * k] : (uint8_t)0;
                __syncwarp();
#pragma unroll
                for (int k = 0; k < 10; ++k) if (lane + 32 * k < nl + nd) W->lens[lane + 32 * k] = t[k];
                __syncwarp();
                if (W->lens[256] == 0) return -10;
            }
            const int brc = infw_build(T, W, nl, nd, lane, type == 1);
            if (brc) return brc;
            {
                uint32_t bp = b.rw * 32u - (uint32_t)b.cnt;
                uint32_t thr = (b.next_line - 2u) << 10;
                const uint32_t *ring = W->ring;
                const uint32_t lane_sh = 8u + 8u * (uint32_t)(lane < 2 ? lane : 2);
                uint16_t *out_lane = o16 + lane;
                int status = 0;
                do {
                    while (bp >= thr) {
                        const uint32_t w = b.next_line * 32u + (uint32_t)lane;
                        const uint32_t v = w < b.nwords ? __ldg(b.words + w) : 0u;
                        W->ring[w & 127u] = v;
                        if ((w & 127u) == 0u) W->ring[128] = v;
                        ++b.next_line;
                        thr += 1024u;
                        __syncwarp();
                    }
                    const uint32_t i0 = (bp >> 5) & 127u;
                    const uint32_t win = __funnelshift_r(ring[i0], ring[i0 + 1], bp);
                    uint32_t e = W->ltab[win & ((1u << INFW_LBITS) - 1u)];
                    if (e == 0) {
                        int cl = 0;
                        const int sym = canon_decode(win, W->lcount, W->lsym, INF_MAXBITS, &cl);
                        e = sym < 0 ? (1u | (3u << 4)) : lit_entry(T, sym, cl);
                    }
                    const uint32_t nb = e & 15u, kind = e & 0x30u;
                    bp += nb;
                    if (kind == 0) {
                        const uint32_t c1 = (e >> 6) & 3u;
                        if (n_out + c1 < cap) {
                            if ((uint32_t)lane <= c1) out_lane[n_out] = (uint16_t)((e >> lane_sh) & 0xFFu);
                            n_out += c1 + 1u;
                        } else {
                            status = -14;
                        }
                    } else if (kind == 0x10u) {
                        const uint32_t xb = e >> 24;
                        const uint32_t len = ((e >> 8) & 0xFFFFu) + ((win >> nb) & ~(0xFFFFFFFFu << xb));
                        bp += xb;
                        const uint32_t j0 = (bp >> 5) & 127u;
                        const uint32_t win2 = __funnelshift_r(ring[j0], ring[j0 + 1], bp);
                        uint32_t d = W->dtab[win2 & ((1u << INFW_DBITS) - 1u)];
                        if (d == 0) {
                            int cl = 0;
                            const int ds = canon_decode(win2, W->dcount, W->dsym, INF_MAXBITS, &cl);
                            d = ds < 0 ? (1u | (15u << 4)) : dist_entry(T, ds, cl);
                        }
                        const uint32_t db = d & 15u, dx = (d >> 4) & 15u;
                        const uint32_t dist = (d >> 8) + ((win2 >> db) & ~(0xFFFFFFFFu << dx));
                        bp += db + dx;
                        // (a distance reaches at most GZ_WIN back: into the place holders, never out of the region)
                        if (dx != 15u && dist <= GZ_WIN && n_out + len <= cap) {
                            __syncwarp();
                            const uint16_t *from = out_lane + n_out - dist;
                            if (dist >= len) {
                                if (len <= 32) {
                                    if ((uint32_t)lane < len) out_lane[n_out] = __ldcg(from);
                                } else {
                                    for (uint32_t i = 0; i + lane < len; i += 32) out_lane[n_out + i] = __ldcg(from + i);
                                }
                            } else {
                                for (uint32_t i = lane; i < len; i += 32) o16[n_out + i] = __ldcg(o16 + n_out - dist + i % dist);
                            }
                            n_out += len;
                        } else {
                            status = -17;
                        }
                    } else {
                        status = kind == 0x20u ? 1 : -15;
                    }
                } while (status == 0);
                if (status != 1) return status;
                b.rw = bp >> 5;
                b.buf = (uint64_t)(W->ring[b.rw & 127u] >> (bp & 31u));
                b.cnt = 32 - (int)(bp & 31u);
                ++b.rw;
            }
        } else {
            return -20;
        }
        // ---- a block has ended: the stream's last, on a later chunk's start, or neither
        const uint32_t pos = b.rw * 32u - (uint32_t)b.cnt;
        res->n_sym = n_out;
        res->end_bit = pos;
        if (pos > a.n_words * 32u) return -19;
        if (last) { res->flags = 1; return 0; }
        if (pos >= next_start) {
            const uint32_t j = gz_lower_bound(a.starts, self + 1, a.n_chunks, pos);
            if (j < a.n_chunks && a.starts[j] == pos) { res->land = j; return 0; }
        }
        if (pos - start_bit > a.max_span_bits) return -23;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(INFW_WARPS * 32, 11)
k_gz_decode(const __grid_constant__ GzDecodeArgs a)
{
    __shared__ InfShared S;
    if (threadIdx.x == 0) {
        const unsigned short lb[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
        const unsigned short le[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
        const unsigned short db[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
        const unsigned short de[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
        const unsigned char od[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        for (int i = 0; i < 29; ++i) { S.T.lbase[i] = lb[i]; S.T.lext[i] = le[i]; }
        for (int i = 0; i < 30; ++i) { S.T.dbase[i] = db[i]; S.T.dext[i] = de[i]; }
        for (int i = 0; i < 19; ++i) S.T.order[i] = od[i];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t warps_total = gridDim.x * INFW_WARPS;
    for (uint32_t i = blockIdx.x * INFW_WARPS + warp; i < a.n_decode; i += warps_total) {
        GzChunkRes r;
        r.n_sym = 0; r.land = GZ_NONE; r.end_bit = 0; r.flags = 0; r.start_bit = a.starts[i]; r.pad[0] = r.pad[1] = r.pad[2] = 0;
        const int rc = gz_chunk_warp(&S, &S.w[warp], a, i, lane, &r);
        if (rc != 0) { r.flags = 2u | ((uint32_t)(-rc) << 8); r.land = GZ_NONE; }      // (the reason travels along for traces)
        if (lane == 0) a.res[i] = r;
        __syncwarp();
    }
}

// What the chain found.
struct GzChainOut {
    uint32_t n_live;         // chunks visited
    uint32_t end_kind;       // 0 = stopped in front of a chunk that starts at or beyond limit_bit (the next segment's true start),
                             // 1 = the stream's final block, 2 = a chunk that failed (the host carries on from its start)
    uint32_t end_bit;        // kind 0 / 2: that chunk's start; kind 1: the bit after the final block
    uint32_t reserved;
    unsigned long long total_text;
};

// One block.  live[k] = k-th visited chunk, text_off[k] = where its text starts (text_off[n_live] = total), win_store
// (n_chunks x GZ_WIN bytes) = its incoming window; out_window = the window after the last visited chunk.
// The walk is serial (a chunk's window comes from its predecessor's), so nothing it needs may be waited for: the
// result record of the chunk after next and the last GZ_WIN symbols of the next chunk are requested before the current
// chunk's window is computed (two symbols per register, thread t owns window positions 2t, 2t+1 + 2048 j).
__device__ __forceinline__ GzChunkRes gz_res_or_none(const GzChunkRes *res, uint32_t c, uint32_t n_chunks)
{
    GzChunkRes r;
    r.n_sym = 0; r.land = GZ_NONE; r.end_bit = 0; r.flags = 2u; r.start_bit = 0xFFFFFFFFu; r.pad[0] = r.pad[1] = r.pad[2] = 0;
    if (c < n_chunks) r = res[c];
    return r;
}

__device__ __forceinline__ void gz_tail_load(const uint16_t *sym, uint32_t n, uint32_t v[16])
{
    // the last GZ_WIN symbols of a chunk of n >= GZ_WIN symbols, two per register; 32-bit loads (the pair straddles two
    // words when the tail starts at an odd symbol)
    const uint16_t *p = sym + (n - GZ_WIN) + 2u * threadIdx.x;
    if (((n - GZ_WIN) & 1u) == 0u) {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(p);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = q[1024 * j];
    } else {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(p - 1);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __funnelshift_r(q[1024 * j], q[1024 * j + 1], 16);
    }
}

__global__ void __launch_bounds__(1024)
k_gz_chain(const GzChunkRes *res, const uint32_t *starts, uint32_t n_chunks, const uint16_t *out16, uint32_t cap, uint32_t limit_bit,
           const uint8_t *first_window, uint32_t *live, unsigned long long *text_off, uint8_t *win_store, uint8_t *out_window,
           GzChainOut *out)
{
    extern __shared__ __align__(16) uint8_t wins[];       // two windows
    uint8_t *cur = wins, *nxt = wins + GZ_WIN;
    for (uint32_t i = threadIdx.x; i < GZ_WIN / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(cur)[i] = reinterpret_cast<const uint4 *>(first_window)[i];
    __syncthreads();
    const size_t region = (size_t)GZ_WIN + cap;
    uint32_t c = 0, k = 0, kind = 2, end_bit = 0, why = 0;
    unsigned long long off = 0;
    GzChunkRes r = gz_res_or_none(res, 0, n_chunks);
    GzChunkRes r2 = gz_res_or_none(res, (r.flags & 3u) ? GZ_NONE : r.land, n_chunks);
    uint32_t v[16], v2[16];
    bool have_v = !(r.flags & 2u) && r.n_sym >= GZ_WIN;
    if (have_v) gz_tail_load(out16 + GZ_WIN, r.n_sym, v);
    for (;;) {
        if (c >= n_chunks) { kind = 2; end_bit = 0; break; }      // (cannot happen: a landing is a chunk index)
        // (a landing spot beyond the limit is not decoded: its record says 0xFFFFFFFF and its start comes from the list)
        if (c != 0 && r.start_bit >= limit_bit) { kind = 0; end_bit = starts[c]; break; }
        const uint32_t sb = r.start_bit;
        if (r.flags & 2u) { kind = 2; end_bit = sb; why = r.flags >> 8; break; }
        // ---- ask for what the next two steps need
        const bool next_valid = !(r.flags & 1u) && r.land < n_chunks;
        const uint32_t c2 = r.land;
        GzChunkRes r3 = gz_res_or_none(res, (next_valid && !(r2.flags & 3u)) ? r2.land : GZ_NONE, n_chunks);
        const bool have_v2 = next_valid && !(r2.flags & 2u) && r2.n_sym >= GZ_WIN && r2.start_bit < limit_bit;
        if (have_v2) gz_tail_load(out16 + (size_t)c2 * region + GZ_WIN, r2.n_sym, v2);
        // ---- this chunk
        if (threadIdx.x == 0) { live[k] = c; text_off[k] = off; }
        uint8_t *ws = win_store + (size_t)k * GZ_WIN;
        for (uint32_t i = threadIdx.x; i < GZ_WIN / 16; i += blockDim.x)
            reinterpret_cast<uint4 *>(ws)[i] = reinterpret_cast<const uint4 *>(cur)[i];
        const uint32_t n = r.n_sym;
        if (have_v) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const uint32_t s0 = v[j] & 0xFFFFu, s1 = v[j] >> 16;
                uint32_t b0 = s0, b1 = s1;
                if (v[j] & 0xFF00FF00u) {                         // (two literals need no look-up)
                    if (s0 >= 256u) b0 = cur[(s0 - 256u) & (GZ_WIN - 1u)];
                    if (s1 >= 256u) b1 = cur[(s1 - 256u) & (GZ_WIN - 1u)];
                }
                *reinterpret_cast<uint16_t *>(nxt + 2u * threadIdx.x + 2048u * j) = (uint16_t)(b0 | (b1 << 8));
            }
        } else {
            // a chunk shorter than the window: the last GZ_WIN bytes of (window ++ chunk)
            const uint16_t *sym = out16 + (size_t)c * region + GZ_WIN;
            for (uint32_t i = threadIdx.x; i < GZ_WIN; i += blockDim.x) {
                const unsigned long long q = (unsigned long long)n + i;
                uint8_t b;
                if (q < GZ_WIN) b = cur[q];
                else {
                    const uint32_t s = sym[q - GZ_WIN];
                    b = s < 256u ? (uint8_t)s : cur[(s - 256u) & (GZ_WIN - 1u)];
                }
                nxt[i] = b;
            }
        }
        __syncthreads();
        uint8_t *t = cur; cur = nxt; nxt = t;
        off += n;
        ++k;
        if (r.flags & 1u) { kind = 1; end_bit = r.end_bit; break; }
        if (!next_valid) { kind = 2; end_bit = sb; --k; off -= n; break; }    // (a chunk without landing is a failed chunk)
        c = c2;
        r = r2;
        r2 = r3;
        have_v = have_v2;
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = v2[j];
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < GZ_WIN / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(out_window)[i] = reinterpret_cast<const uint4 *>(cur)[i];
    if (threadIdx.x == 0) {
        text_off[k] = off;
        out->n_live = k; out->end_kind = kind; out->end_bit = end_bit; out->reserved = why; out->total_text = off;
    }
}

// Pieces of GZ_PIECE bytes of text: symbols -> bytes (place holders through the chunk's window), newlines per piece.
// hist0 = bytes of real text in front of the segment (at most GZ_WIN): a place holder p of visited chunk k stands for the
// byte GZ_WIN - p before the chunk, which exists only when GZ_WIN - p <= hist0 + text_off[k].
#define GZ_PIECE 65536u
__global__ void __launch_bounds__(256)
k_gz_resolve(const uint32_t *live, const unsigned long long *text_off, uint32_t n_live, const uint16_t *out16, uint32_t cap,
             const uint8_t *win_store, uint8_t *text, uint32_t *piece_nl, uint32_t hist0, uint32_t *flag_unknown)
{
    __shared__ uint32_t s_nl;
    const unsigned long long lo = (unsigned long long)blockIdx.x * GZ_PIECE;
    const unsigned long long total = text_off[n_live];
    const unsigned long long hi = lo + GZ_PIECE < total ? lo + GZ_PIECE : total;
    if (threadIdx.x == 0) s_nl = 0;
    __syncthreads();
    // first visited chunk that overlaps [lo, hi)
    uint32_t a = 0, b = n_live;
    while (a + 1 < b) {
        const uint32_t mid = (a + b) >> 1;
        if (text_off[mid] <= lo) a = mid; else b = mid;
    }
    uint32_t nl = 0, unknown = 0;
    for (uint32_t k = a; k < n_live && text_off[k] < hi; ++k) {
        const unsigned long long c_lo = text_off[k], c_hi = text_off[k + 1];
        const unsigned long long from = c_lo > lo ? c_lo : lo, to = c_hi < hi ? c_hi : hi;
        const uint16_t *sym = out16 + (size_t)live[k] * (GZ_WIN + (size_t)cap) + GZ_WIN;
        const uint8_t *win = win_store + (size_t)k * GZ_WIN;
        const unsigned long long hist = hist0 + c_lo;
        const uint32_t n_invalid = hist >= GZ_WIN ? 0u : GZ_WIN - (uint32_t)hist;    // place holders below this point before the stream
        for (unsigned long long q = from + threadIdx.x; q < to; q += blockDim.x) {
            const uint32_t s = sym[q - c_lo];
            uint8_t v;
            if (s < 256u) v = (uint8_t)s;
            else {
                v = __ldg(win + ((s - 256u) & (GZ_WIN - 1u)));
                if (s - 256u < n_invalid) unknown = 1;
            }
            text[q] = v;
            nl += v == (uint8_t)'\n';
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { nl += __shfl_xor_sync(0xffffffffu, nl, o); unknown |= __shfl_xor_sync(0xffffffffu, unknown, o); }
    if ((threadIdx.x & 31) == 0) { if (nl) atomicAdd(&s_nl, nl); if (unknown) atomicOr(flag_unknown, 1u); }
    __syncthreads();
    if (threadIdx.x == 0) piece_nl[blockIdx.x] = s_nl;
}

// CRC-32 of pieces of GZ_CRC_PIECE bytes, one thread each (the host combines them with zlib's combine operator).
#define GZ_CRC_PIECE 16384u
__global__ void __launch_bounds__(128)
k_gz_crc(const uint8_t *text, unsigned long long total, uint32_t *piece_crc)
{
    __shared__ uint32_t tab[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        uint32_t c = (uint32_t)i;
        for (int k = 0; k < 8; ++k) c = (c & 1u) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
        tab[i] = c;
    }
    __syncthreads();
    const unsigned long long piece = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long lo = piece * GZ_CRC_PIECE;
    if (lo >= total) return;
    const unsigned long long hi = lo + GZ_CRC_PIECE < total ? lo + GZ_CRC_PIECE : total;
    uint32_t crc = 0xFFFFFFFFu;
    unsigned long long i = lo;
    // (text is 16-byte aligned and lo a multiple of 16)
    for (; i + 16 <= hi; i += 16) {
        const uint4 w = __ldg(reinterpret_cast<const uint4 *>(text + i));
        uint32_t x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t v = x[j];
#pragma unroll
            for (int k = 0; k < 4; ++k) { crc = tab[(crc ^ v) & 0xFFu] ^ (crc >> 8); v >>= 8; }
        }
    }
    for (; i < hi; ++i) crc = tab[(crc ^ text[i]) & 0xFFu] ^ (crc >> 8);
    piece_crc[piece] = crc ^ 0xFFFFFFFFu;
}

// d_list: scratch for the offsets that pass the first test (list_cap + 1 words; the last one is the counter)
int launch_gz_search(const uint32_t *d_z32, uint32_t n_words, uint32_t lo_bit, uint32_t hi_bit, uint32_t *d_cand, uint32_t *d_n_cand,
                     uint32_t cand_cap, uint32_t *d_list, uint32_t list_cap, cudaStream_t st)
{
    if (hi_bit <= lo_bit) return VFB_OK;
    VFB_CUDA(cudaMemsetAsync(d_list + list_cap, 0, 4, st));
    k_gz_search1<<<148 * 8, 256, 0, st>>>(d_z32, n_words, lo_bit, hi_bit, d_list, d_list + list_cap, list_cap);
    k_gz_search2<<<148 * 8, 128, 0, st>>>(d_z32, n_words, d_list, d_list + list_cap, list_cap, d_cand, d_n_cand, cand_cap);
    g_launches += 2;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

int launch_gz_decode(const uint32_t *d_z32, uint32_t n_words, const uint32_t *d_starts, uint32_t n_chunks, uint32_t n_decode,
                     uint16_t *d_out16, uint32_t cap, uint32_t max_span_bits, void *d_res, cudaStream_t st)
{
    if (n_decode == 0) return VFB_OK;
    GzDecodeArgs a{d_z32, n_words, d_starts, n_chunks, n_decode, d_out16, cap, max_span_bits, static_cast<GzChunkRes *>(d_res)};
    uint32_t blocks = (n_decode + INFW_WARPS - 1) / INFW_WARPS;
    if (blocks > 148u * 11u) blocks = 148u * 11u;
    k_gz_decode<<<blocks, INFW_WARPS * 32, 0, st>>>(a);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

int launch_gz_chain(const void *d_res, const uint32_t *d_starts, uint32_t n_chunks, const uint16_t *d_out16, uint32_t cap,
                    uint32_t limit_bit, const uint8_t *d_first_window, uint32_t *d_live, unsigned long long *d_text_off,
                    uint8_t *d_win_store, uint8_t *d_out_window, void *d_out, cudaStream_t st)
{
    static bool attr = false;
    if (!attr) {
        VFB_CUDA(cudaFuncSetAttribute(k_gz_chain, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * GZ_WIN)));
        attr = true;
    }
    k_gz_chain<<<1, 1024, 2 * GZ_WIN, st>>>(static_cast<const GzChunkRes *>(d_res), d_starts, n_chunks, d_out16, cap, limit_bit,
                                            d_first_window, d_live, d_text_off, d_win_store, d_out_window,
                                            static_cast<GzChainOut *>(d_out));
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

int launch_gz_resolve(const uint32_t *d_live, const unsigned long long *d_text_off, uint32_t n_live, unsigned long long total_text,
                      const uint16_t *d_out16, uint32_t cap, const uint8_t *d_win_store, uint8_t *d_text, uint32_t *d_piece_nl,
                      uint32_t *d_piece_crc, uint32_t hist, uint32_t *d_flag_unknown, cudaStream_t st)
{
    if (total_text == 0) return VFB_OK;
    const uint32_t pieces = (uint32_t)((total_text + GZ_PIECE - 1) / GZ_PIECE);
    k_gz_resolve<<<pieces, 256, 0, st>>>(d_live, d_text_off, n_live, d_out16, cap, d_win_store, d_text, d_piece_nl,
                                         hist, d_flag_unknown);
    const uint32_t cp = (uint32_t)((total_text + GZ_CRC_PIECE - 1) / GZ_CRC_PIECE);
    k_gz_crc<<<(cp + 127) / 128, 128, 0, st>>>(d_text, total_text, d_piece_crc);
    g_launches += 2;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

int launch_inflate(const uint8_t *d_z, const vfb_member *d_members, uint32_t n_members, uint8_t *d_out,
                   uint32_t *d_first_bad, cudaStream_t st)
{
    if (n_members == 0) return VFB_OK;
    const InflateArgs a{d_z, d_members, n_members, d_out, d_first_bad};
    static int bps = 0, sms = 0;
    if (!bps) {
        int dev = 0;
        VFB_CUDA(cudaGetDevice(&dev));
        VFB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        VFB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_inflate_warp, INFW_WARPS * 32, 0));
        if (bps < 1) bps = 1;
    }
    uint32_t blocks = (n_members + INFW_WARPS - 1) / INFW_WARPS;
    if (blocks > (uint32_t)(sms * bps)) blocks = (uint32_t)(sms * bps);
    k_inflate_warp<<<blocks, INFW_WARPS * 32, 0, st>>>(a);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

}  // namespace vfb
