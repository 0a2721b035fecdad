"""A deflate writer for tests (RFC 1951 / 1952): streams made from explicit choices, not from compression heuristics.

zlib's encoder never makes some legal choices (a code-length run across the literal/length - distance boundary, 258 as
code 284 with 31 extra bits, 15-bit codes, a distance code of one 1-bit code, stored blocks at every bit phase, ...) and
never writes an invalid header.  This module writes both, so that the decoders can be held to what zlib accepts and
rejects.  Every `Deflate` records the features it used (`.features`), so a test can assert coverage.

Tokens: an int 0..255 is a literal; (length, dist) is a match; (258, dist, True) writes 258 as code 284 + 31 extra bits.
Raw symbols for broken fixed blocks: ("lsym", s) writes literal/length symbol s, ("dsym", length, s) a match whose
distance symbol is s (no extra bits).

`Deflate.text` is what a decoder outputs when it reads zeros for every byte before the stream's first one: the true text
of a legal stream, and the output a lenient decoder would check the trailer against in an invalid one.
"""
import struct
import zlib

WSIZE = 32768
LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEXT = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
         6145, 8193, 12289, 16385, 24577]
DEXT = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32


class BitWriter:
    """LSB-first bit packing (RFC 1951 3.1.1)."""

    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    @property
    def nbits(self):
        return len(self.out) * 8 + self.n

    def put(self, value, n):
        assert 0 <= value < (1 << n) or n == 0 and value == 0, (value, n)
        self.acc |= value << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8

    def put_code(self, code, length):
        """A Huffman code, most significant bit first."""
        r = 0
        for b in range(length):
            r |= ((code >> b) & 1) << (length - 1 - b)
        self.put(r, length)

    def getvalue(self):
        return bytes(self.out) + (bytes([self.acc]) if self.n else b"")


def kraft(lengths):
    """Sum of 2^-l over the nonzero lengths, in units of 2^-15."""
    return sum(1 << (15 - l) for l in lengths if l)


def canonical_codes(lengths):
    """RFC 1951 3.2.2.  Over-subscribed lengths get codes too (wrapped to their length): only a broken case uses them."""
    maxl = max(lengths) if lengths else 0
    bl_count = [0] * (maxl + 2)
    for l in lengths:
        if l:
            bl_count[l] += 1
    code, nxt = 0, [0] * (maxl + 2)
    for bits in range(1, maxl + 1):
        code = (code + bl_count[bits - 1]) << 1
        nxt[bits] = code
    codes = [0] * len(lengths)
    for s, l in enumerate(lengths):
        if l:
            codes[s] = nxt[l] & ((1 << l) - 1)
            nxt[l] += 1
    return codes


def limited_lengths(freqs, limit):
    """Optimal length-limited Huffman code lengths (package-merge) for the symbols with freqs[s] > 0.  One used symbol
    gets length 1 (the only incomplete code RFC 1951 / zlib allow)."""
    used = [s for s, f in enumerate(freqs) if f > 0]
    lens = [0] * len(freqs)
    if not used:
        return lens
    if len(used) == 1:
        lens[used[0]] = 1
        return lens
    assert len(used) <= (1 << limit)
    leaves = sorted((freqs[s], (s,)) for s in used)
    items = list(leaves)
    for _ in range(limit - 1):
        merged = [(items[i][0] + items[i + 1][0], items[i][1] + items[i + 1][1]) for i in range(0, len(items) - 1, 2)]
        items = sorted(leaves + merged, key=lambda t: t[0])
    for _, syms in items[:2 * len(used) - 2]:
        for s in syms:
            lens[s] += 1
    assert max(lens) <= limit and kraft(lens) == 1 << 15
    return lens


def len_symbol(length, as284=False):
    """(symbol, extra bits, extra value) of a match length."""
    assert 3 <= length <= 258
    if length == 258 and not as284:
        return 285, 0, 0
    i = max(k for k in range(28) if LBASE[k] <= length)
    assert length - LBASE[i] < (1 << LEXT[i])
    return 257 + i, LEXT[i], length - LBASE[i]


def dist_symbol(dist):
    assert 1 <= dist <= WSIZE
    i = max(k for k in range(30) if DBASE[k] <= dist)
    return i, DEXT[i], dist - DBASE[i]


def lz77(buf, start, max_len=258, max_dist=WSIZE, min_len=3):
    """Greedy tokens for buf[start:], matches may reach into buf[:start] (the text of earlier blocks)."""
    last = {}
    for p in range(max(0, start - max_dist), start):
        last[bytes(buf[p:p + 3])] = p
    toks, i, n = [], start, len(buf)
    while i < n:
        key = bytes(buf[i:i + 3])
        j = last.get(key)
        best = 0
        if j is not None and i - j <= max_dist and len(key) == 3:
            m = 0
            while m < max_len and i + m < n and buf[j + m] == buf[i + m]:
                m += 1
            best = m
        if best >= min_len:
            toks.append((best, i - j))
            for p in range(i, min(i + best, n - 2)):
                last[bytes(buf[p:p + 3])] = p
            i += best
        else:
            toks.append(buf[i])
            last[key] = i
            i += 1
    return toks


def rle_lengths(seq, lo=0, hi=None):
    """zlib-style run-length code of seq[lo:hi] as (symbol, extra bits, extra value): 16 repeats the previous length 3-6
    times, 17 writes 3-10 zeros, 18 11-138 zeros."""
    hi = len(seq) if hi is None else hi
    out, i = [], lo
    while i < hi:
        v, r = seq[i], 1
        while i + r < hi and seq[i + r] == v:
            r += 1
        if v == 0:
            left = r
            while left >= 11:
                k = min(left, 138)
                out.append((18, 7, k - 11))
                left -= k
            if left >= 3:
                out.append((17, 3, left - 3))
                left = 0
            out += [(0, 0, 0)] * left
        else:
            out.append((v, 0, 0))
            left = r - 1
            while left >= 3:
                k = min(left, 6)
                out.append((16, 2, k - 3))
                left -= k
            out += [(v, 0, 0)] * left
        i += r
    return out


def cl_runs(cl_syms):
    """(first index, count, symbol) of every code-length symbol."""
    out, idx = [], 0
    for s, nb, v in cl_syms:
        c = 1 if s < 16 else (3 + v if s in (16, 17) else 11 + v)
        out.append((idx, c, s))
        idx += c
    return out


class Deflate:
    """One raw deflate stream, block by block."""

    def __init__(self):
        self.w = BitWriter()
        self.buf = bytearray(WSIZE)        # zeros stand for the bytes before the stream
        self.features = set()
        self.final_written = False

    @property
    def text(self):
        return bytes(self.buf[WSIZE:])

    @property
    def phase(self):
        return self.w.nbits % 8

    def getvalue(self):
        return self.w.getvalue()

    def raw(self, value, n):
        """Raw bits (broken headers)."""
        self.w.put(value, n)

    def tokens_for(self, data, **kw):
        """Greedy LZ77 tokens for `data` as the continuation of the text so far."""
        buf = self.buf[WSIZE:] + data
        return lz77(buf, len(buf) - len(data), **kw)

    # ---- token bookkeeping
    def _apply(self, tok):
        if isinstance(tok, int):
            self.buf.append(tok)
            return
        if tok[0] in ("lsym", "dsym"):
            self.features.add("raw_symbol")
            if tok[0] == "dsym":
                for _ in range(tok[1]):
                    self.buf.append(0)
            return
        length, dist = tok[0], tok[1]
        if dist > len(self.buf) - WSIZE:
            self.features.add("too_far_back")
        if dist == WSIZE:
            self.features.add("dist_32768")
        if dist < length:
            self.features.add("overlap_copy")
        if length == 258:
            self.features.add("len258_code284" if len(tok) > 2 and tok[2] else "len258_code285")
        for _ in range(length):
            self.buf.append(self.buf[-dist])

    def _symbols(self, tokens):
        """(lit symbol, extra n, extra v, dist symbol or None, extra n, extra v) per token."""
        out = []
        for t in tokens:
            if isinstance(t, int):
                out.append((t, 0, 0, None, 0, 0))
            elif t[0] == "lsym":
                out.append((t[1], 0, 0, None, 0, 0))
            elif t[0] == "dsym":
                s, n, v = len_symbol(t[1])
                out.append((s, n, v, t[2], 0, 0))
            else:
                s, n, v = len_symbol(t[0], len(t) > 2 and t[2])
                d, dn, dv = dist_symbol(t[1])
                out.append((s, n, v, d, dn, dv))
        return out

    def _write_tokens(self, syms, lit_lens, dist_lens, tokens):
        lc, dc = canonical_codes(lit_lens), canonical_codes(dist_lens)
        for (s, n, v, d, dn, dv), t in zip(syms, tokens):
            l = lit_lens[s] if s < len(lit_lens) else 0
            assert l, "literal/length symbol %d has no code" % s
            self.w.put_code(lc[s], l)
            self.w.put(v, n)
            self.features.add("lit_code_len_%d" % l)
            if d is not None:
                dl = dist_lens[d] if d < len(dist_lens) else 0
                assert dl, "distance symbol %d has no code" % d
                self.w.put_code(dc[d], dl)
                self.w.put(dv, dn)
                self.features.add("dist_code_len_%d" % dl)
            self._apply(t)
        if len(lit_lens) > 256 and lit_lens[256]:
            self.w.put_code(lc[256], lit_lens[256])

    def _header(self, final, btype):
        assert not self.final_written, "a block after the final block"
        self.w.put(1 if final else 0, 1)
        self.w.put(btype, 2)
        self.final_written = final
        if final:
            self.features.add("bfinal")

    # ---- blocks
    def stored(self, payload, final=False, nlen=None, pad_bits=0):
        """A stored block; `pad_bits` fills the bits up to the byte boundary (decoders must ignore them); `nlen`
        overrides NLEN (a broken case)."""
        assert len(payload) <= 65535
        self.features.add("stored")
        if len(payload) in (0, 65535):
            self.features.add("stored_%d_phase_%d" % (len(payload), self.phase))
        self._header(final, 0)
        k = (8 - self.w.n) % 8
        if pad_bits & ((1 << k) - 1):
            self.features.add("stored_pad_bits_set")
        self.w.put(pad_bits & ((1 << k) - 1), k)
        self.w.put(len(payload), 16)
        self.w.put((len(payload) ^ 0xFFFF) if nlen is None else nlen, 16)
        self.w.out += payload                 # (byte aligned here)
        self.buf += payload

    def fixed(self, tokens, final=False):
        self.features.add("fixed")
        self._header(final, 1)
        self._write_tokens(self._symbols(tokens), FIXED_LIT, FIXED_DIST, tokens)

    def goto_phase(self, phase, byte=0xE9):
        """A fixed non-final block of literals with 9-bit codes (bytes 144..255) after which the next block starts at bit
        phase `phase`: 10 + 9 n bits."""
        n = (phase - self.phase - 2) % 8
        self.fixed([byte] * n)

    def dynamic(self, tokens, final=False, *, limit=15, lit_lens=None, dist_lens=None, lit_weights=None, dist_weights=None,
                nlen=None, ndist=None, ncode=None, rle="per_tree", cl_syms=None, cl_lens=None, tamper_codes=None,
                tamper_cl=None, check=True):
        """A dynamic block.  Code lengths are given (lit_lens / dist_lens, indexed by symbol) or built from the tokens'
        symbol counts plus `*_weights` ({symbol: extra count}) as codes limited to `limit` bits.  nlen / ndist / ncode
        (HLIT + 257, HDIST + 1, HCLEN + 4) default to the shortest that hold every nonzero length.  rle: "per_tree"
        (zlib: the two sequences coded separately), "across" (one run-length code over both: runs may cross), "none" (a
        length symbol per length); cl_syms / cl_lens replace the run-length symbols / the code-length code.  check:
        every code complete (or a single 1-bit code) and the header in range, as a legal stream needs.  Broken headers:
        tamper_codes(lit_lens, dist_lens) and tamper_cl(cl_syms, cl_lens) edit the lists in place before they are
        written (with check=False)."""
        self.features.add("dynamic")
        syms = self._symbols(tokens)
        lf, df = [0] * 288, [0] * 32
        for s, _, _, d, _, _ in syms:
            lf[s] += 1
            if d is not None:
                df[d] += 1
        lf[256] += 1
        for s, c in (lit_weights or {}).items():
            lf[s] += c
        for s, c in (dist_weights or {}).items():
            df[s] += c
        if lit_lens is None:
            lit_lens = limited_lengths(lf[:286], limit)
        if dist_lens is None:
            dist_lens = limited_lengths(df[:30], limit)
        lit_lens, dist_lens = list(lit_lens), list(dist_lens)
        if nlen is None:
            nlen = max(257, max((s + 1 for s, l in enumerate(lit_lens) if l), default=0))
        if ndist is None:
            ndist = max(1, max((s + 1 for s, l in enumerate(dist_lens) if l), default=0))
        lit_lens = (lit_lens + [0] * 288)[:max(nlen, len(lit_lens))]
        dist_lens = (dist_lens + [0] * 32)[:max(ndist, len(dist_lens))]
        if tamper_codes:
            tamper_codes(lit_lens, dist_lens)
        seq = lit_lens[:nlen] + dist_lens[:ndist]
        if check:
            assert nlen <= 286 and ndist <= 30 and not any(lit_lens[nlen:]) and not any(dist_lens[ndist:])
            assert lit_lens[256]
            for lens in (lit_lens[:nlen], dist_lens[:ndist]):
                used = [l for l in lens if l]
                assert kraft(lens) == 1 << 15 or used == [1] or not used, lens
        # features of the code
        if nlen == 286:
            self.features.add("hlit_286")
        if not lit_lens[nlen - 1]:
            self.features.add("hlit_trailing_zero")
        if not dist_lens[ndist - 1]:
            self.features.add("hdist_trailing_zero")
        dused = [l for l in dist_lens[:ndist] if l]
        if not dused:
            self.features.add("no_distance_codes")
        elif dused == [1]:
            self.features.add("single_distance_code")
        if [l for l in lit_lens[:nlen] if l] == [1]:
            self.features.add("single_literal_code")
        # the code-length symbols
        if cl_syms is None:
            if rle == "per_tree":
                cl_syms = rle_lengths(seq, 0, nlen) + rle_lengths(seq, nlen, nlen + ndist)
            elif rle == "across":
                cl_syms = rle_lengths(seq)
            else:
                cl_syms = [(l, 0, 0) for l in seq]
        for first, count, s in cl_runs(cl_syms):
            if s >= 16 and first < nlen < first + count:
                self.features.add("rle_across_boundary")
            if s >= 16:
                self.features.add("cl%d_%d" % (s, count))
        if cl_lens is None:
            cf = [0] * 19
            for s, _, _ in cl_syms:
                cf[s] += 1
            if sum(1 for c in cf if c) == 1:          # one symbol: a second one makes the code complete
                cf[0 if not cf[0] else 1] += 1
            cl_lens = limited_lengths(cf, 7)
        cl_lens = list(cl_lens)
        if tamper_cl:
            tamper_cl(cl_syms, cl_lens)
        if ncode is None:
            ncode = max(4, max((i + 1 for i, s in enumerate(ORDER) if cl_lens[s]), default=0))
        if check:
            assert kraft(cl_lens) == 1 << 15 and not any(cl_lens[s] for s in ORDER[ncode:])
        self.features.add("hclen_%d" % ncode)
        # write
        self._header(final, 2)
        self.w.put(nlen - 257, 5)
        self.w.put(ndist - 1, 5)
        self.w.put(ncode - 4, 4)
        for s in ORDER[:ncode]:
            self.w.put(cl_lens[s], 3)
        cc = canonical_codes(cl_lens)
        for s, n, v in cl_syms:
            self.w.put_code(cc[s], cl_lens[s])
            self.w.put(v, n)
        if not syms:
            self.features.add("empty_dynamic")
        before = len(self.buf)
        self._write_tokens(syms, lit_lens, dist_lens, tokens)
        if 0 < len(self.buf) - before < 1024:
            self.features.add("tiny_dynamic")


def gzip_member(deflate, text):
    """A plain gzip member; CRC-32 and ISIZE over `text`."""
    return (b"\x1f\x8b\x08\x00\0\0\0\0\0\xff" + deflate +
            struct.pack("<II", zlib.crc32(text) & 0xFFFFFFFF, len(text) & 0xFFFFFFFF))


def bgzf_member(deflate, text):
    """A block-gzip member: the "BC" extra subfield (2 bytes long) holds the member's size - 1."""
    size = 18 + len(deflate) + 8
    assert size <= 65536 and len(text) <= 65536
    hdr = struct.pack("<BBBBIBBH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6) + b"BC" + struct.pack("<HH", 2, size - 1)
    return hdr + gzip_member(deflate, text)[10:]


def zlib_verdict(deflate):
    """(True, text) when zlib inflates the raw stream to its end, (False, reason) otherwise."""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(deflate) + d.flush()
    except zlib.error as e:
        return False, str(e)
    return (True, out) if d.eof else (False, "incomplete stream")
