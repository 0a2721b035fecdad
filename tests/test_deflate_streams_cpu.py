"""Hand-built deflate streams (tests/deflate_writer.py) through the host decoders: the serial zlib path and the parallel
single-stream gunzip (pgunzip.cu) through vfb_debug_inflate_file.

zlib's encoder never writes some legal choices (code-length runs across the literal/length - distance boundary, 258 as
284 + 31, 15-bit codes, a one-code distance code, stored blocks at every bit phase, many tiny dynamic blocks) and never
writes an invalid header, so the corpus here is written by hand.  What zlib makes of every stream is the verdict: a legal
stream must decode to zlib's output on every path, an invalid one must fail on every path.  Every invalid member carries
the CRC-32 and ISIZE of what a lenient decoder would output (reading zeros before the stream's first byte), so a decoder
that skips the rule under test is not rescued by the trailer check.  The corpus is shared with the device tests
(test_gpu_deflate_streams.py)."""
import ctypes
import functools
import gzip
import random
import struct
from collections import namedtuple

import pytest

from deflate_writer import Deflate, bgzf_member, gzip_member, kraft, lz77, zlib_verdict
from test_pgunzip_cpu import fastq, inflate, normalised

Case = namedtuple("Case", "name deflate text features")


def giant(body):
    """One FASTQ record around arbitrary bytes (the host harness only cuts at 4-line boundaries)."""
    return b"@h\n" + bytes(body).replace(b"\n", b" ").replace(b"\r", b" ") + b"\n+\nq\n"


def _noline(rng, n, alphabet=None):
    if alphabet:
        return bytes(rng.choice(alphabet) for _ in range(n))
    return bytes(rng.randrange(256) for _ in range(n)).replace(b"\n", b" ")


def _around(d, text, k, tok):
    """Tokens for `text` with `tok` put in after its first k bytes (the rest only refers to itself)."""
    return d.tokens_for(text[:k]) + [tok] + lz77(text[k:], 0)


def _case(name, d):
    return Case(name, d.getvalue(), d.text, frozenset(d.features))


@functools.lru_cache(maxsize=None)
def legal_corpus():
    rng = random.Random(1951)
    out = []

    # stored blocks of 0 and 65535 bytes with the block header at every bit phase, the skipped bits set
    for size in (0, 65535):
        d = Deflate()
        d.fixed(list(b"@h\n"))
        for p in range(8):
            d.goto_phase(p)
            d.stored(_noline(rng, size) if size else b"", pad_bits=0x7F)
        d.fixed(list(b"\n+\nq\n"), final=True)
        out.append(_case("stored_%d_every_phase" % size, d))

    # many tiny dynamic blocks mixed with stored, fixed and empty dynamic blocks; matches reach into earlier blocks
    text = fastq(180, rng)
    d = Deflate()
    pos = 0
    while pos < len(text):
        n = min(rng.choice([20, 60, 150, 400]) + rng.randrange(40), len(text) - pos)
        piece, last = text[pos:pos + n], pos + n >= len(text)
        k = rng.randrange(10)
        if k == 0:
            d.dynamic([])
        if k == 1:
            d.stored(piece, final=last)
        elif k == 2:
            d.fixed(d.tokens_for(piece), final=last)
        else:
            d.dynamic(d.tokens_for(piece), final=last)
        pos += n
    out.append(_case("tiny_dynamic_blocks", d))

    # 15-bit codes: exponential weights on unused symbols push the rarely used ones to the limit
    x = _noline(rng, 100, b"klmnopqrstuvwxyz")
    body = x + b"!$%" + _noline(rng, 30000, b"ACGT") + x
    d = Deflate()
    d.dynamic(d.tokens_for(b"@h\n"))
    d.dynamic(d.tokens_for(giant(body)[3:]), final=True, lit_weights={0xC0 + k: 1 << (k + 3) for k in range(26)},
              dist_weights={k: 1 << (k + 1) for k in range(29)})
    out.append(_case("code_length_15", d))

    # code-length runs across the boundary and at their extremes: 18 x 138 (literals 0..138 unused), 17 x 10 (200..209),
    # 16 x 6 (equal lengths), HLIT = 286 and HCLEN = 19 with trailing zeros; then a one-code distance code whose
    # leading zeros run on from the literal/length code's trailing ones
    alpha = bytes(b for b in range(139, 256) if not 200 <= b <= 209)
    d = Deflate()
    d.fixed(list(b"@h\n"))
    d.dynamic(list(_noline(rng, 3000, alpha)), nlen=286, ncode=19, rle="across")
    y = _noline(rng, 300, alpha)
    d.dynamic(d.tokens_for(y + _noline(rng, 2500, alpha) + y), rle="across")
    d.dynamic(d.tokens_for(y), rle="none")
    d.fixed(list(b"\n+\nq\n"), final=True)
    out.append(_case("code_length_runs", d))

    # 258 as 285 and as 284 + 31, overlapping copies, distance 32768 (a window's worth of random bytes, repeated)
    w = _noline(rng, 32768)
    d = Deflate()
    d.dynamic(d.tokens_for(b"@h\n" + b"A" * 3000))
    d.dynamic([(t[0], t[1], True) if isinstance(t, tuple) and t[0] == 258 else t for t in d.tokens_for(b"C" * 3000)])
    d.dynamic(d.tokens_for(w))
    d.dynamic(d.tokens_for(w[:5000]))
    d.fixed(d.tokens_for(w[5000:9000]))
    d.dynamic(d.tokens_for(b"\n+\nq\n"), final=True)
    out.append(_case("long_matches", d))

    # a one-code distance code (every match at distance 1), no distance codes at all, empty dynamic blocks
    text = fastq(120, rng, qual="FFFFFFFFFFFFF#")
    cut = text.find(b"\n@", len(text) // 2) + 1
    d = Deflate()
    d.dynamic(d.tokens_for(text[:cut], max_dist=1))
    d.dynamic([])
    d.dynamic(list(text[cut:]))
    d.dynamic([], final=True)
    out.append(_case("one_code_and_no_codes", d))

    # zlib-like blocks of a larger FASTQ file: per-tree run-length codes, every block boundary a place to start from
    text = fastq(900, rng)
    d = Deflate()
    for i in range(0, len(text), 16000):
        d.dynamic(d.tokens_for(text[i:i + 16000]), final=i + 16000 >= len(text))
    out.append(_case("fastq_blocks", d))
    return out


def _lead(d, rng, n=40):
    """A legal non-final dynamic block of FASTQ records."""
    d.dynamic(d.tokens_for(fastq(n, rng)))


def _finish(d, rng, n=10):
    d.dynamic(d.tokens_for(fastq(n, rng)), final=True)


@functools.lru_cache(maxsize=None)
def invalid_corpus():
    rng = random.Random(1952)
    out = []

    def build(name, broken, lead=True, finish=True):
        d = Deflate()
        if lead:
            _lead(d, rng)
        broken(d)
        if finish:
            _finish(d, rng)
        out.append(_case(name, d))
        return d

    recs = lambda n=20: fastq(n, rng)

    def unused(lens, limit=None):
        return next(s for s in range(len(lens) if limit is None else limit) if not lens[s])

    # over-subscribed codes: one more code of the longest length
    build("cl_code_oversubscribed", lambda d: d.dynamic(d.tokens_for(recs()), ncode=19, check=False,
          tamper_cl=lambda syms, cl: cl.__setitem__(unused(cl), max(cl))))
    build("lit_code_oversubscribed", lambda d: d.dynamic(d.tokens_for(recs()), check=False,
          tamper_codes=lambda ll, dl: ll.__setitem__(unused(ll, 256), max(ll))))
    build("dist_code_oversubscribed", lambda d: d.dynamic(d.tokens_for(recs()), check=False, ndist=30,
          tamper_codes=lambda ll, dl: dl.__setitem__(unused(dl, 30), max(dl))))

    # an incomplete code-length code: its longest code one bit longer (still a prefix code)
    def lengthen(syms, cl):
        s = max((s for s in range(19) if 0 < cl[s] < 7), key=lambda s: cl[s])
        cl[s] += 1
    build("cl_code_incomplete", lambda d: d.dynamic(d.tokens_for(recs()), ncode=19, check=False, tamper_cl=lengthen))

    # a single code of length >= 2: the literal/length code of an empty block, the distance code of distance-1 matches
    for n in (2, 3):
        build("lit_single_code_len%d" % n, lambda d, n=n: d.dynamic([], check=False, lit_lens=[0] * 256 + [n]))
        build("dist_single_code_len%d" % n, lambda d, n=n: d.dynamic(d.tokens_for(fastq(20, rng, "FFFFFFFF#"),
                                                                                  max_dist=1),
                                                                     check=False, dist_lens=[n]))

    # no end-of-block code; 16 with nothing to repeat; a repeat past HLIT + HDIST; HCLEN = 4 (no length can be nonzero)
    build("no_end_of_block_code", lambda d: d.dynamic(d.tokens_for(recs()), check=False,
          tamper_codes=lambda ll, dl: ll.__setitem__(256, 0)))

    def first_16(d):
        toks = d.tokens_for(recs())
        def tamper(syms, cl):
            assert cl[16]
            syms.insert(0, (16, 2, 0))
        d.dynamic(toks, check=False, tamper_cl=tamper)
    build("repeat_with_nothing_to_repeat", first_16)

    def overrun(syms, cl):
        assert cl[18]
        syms[-1] = (18, 7, 127)
    build("repeat_past_the_end", lambda d: d.dynamic(d.tokens_for(recs()), check=False, ncode=19, tamper_cl=overrun))
    build("hclen_4", lambda d: d.dynamic([], check=False, ncode=4, cl_syms=[(18, 7, 127), (18, 7, 109)],
                                         cl_lens=[1] + [0] * 15 + [0, 2, 2], lit_lens=[0] * 257, dist_lens=[0]))

    # HLIT / HDIST out of range (the codes themselves complete)
    for nlen in (287, 288):
        build("hlit_%d" % nlen, lambda d, nlen=nlen: d.dynamic(d.tokens_for(recs()), check=False, nlen=nlen))
    for ndist in (31, 32):
        build("hdist_%d" % ndist, lambda d, ndist=ndist: d.dynamic(d.tokens_for(recs()), check=False, ndist=ndist))

    # symbols a fixed block must not use
    for name, tok in (("fixed_lit_286", ("lsym", 286)), ("fixed_lit_287", ("lsym", 287)),
                      ("fixed_dist_30", ("dsym", 5, 30)), ("fixed_dist_31", ("dsym", 5, 31))):
        build(name, lambda d, tok=tok: d.fixed(_around(d, recs(8), 700, tok)))

    build("stored_nlen_mismatch", lambda d: d.stored(recs(5), nlen=0x1234))
    build("btype_3", lambda d: (d.raw(0, 1), d.raw(3, 2), d.raw(0x5A5A, 16)))
    build("no_final_block", lambda d: d.dynamic(d.tokens_for(recs())), finish=False)

    # truncated inside a dynamic header and inside stored data (the member ends there: no trailer)
    d = Deflate()
    _lead(d, rng)
    cut = len(d.getvalue())
    d.dynamic(d.tokens_for(recs()), final=True)
    out.append(Case("truncated_in_dynamic_header", d.getvalue()[:cut + 20], d.text, frozenset(d.features | {"truncated"})))
    d = Deflate()
    _lead(d, rng)
    d.stored(recs(10), final=True)
    out.append(Case("truncated_in_stored_data", d.getvalue()[:-200], d.text, frozenset(d.features | {"truncated"})))

    # a distance too far back: in the first block; in a later non-final dynamic block after ~4 KB of text (on the
    # device: a chunk after the first); after ~500 bytes of text, in a block larger than a small device chunk (zlib
    # takes that one over with the text so far as its dictionary, and must not be given more)
    def far_first(d):
        t = recs(3)
        d.dynamic(_around(d, t, 10, (20, 40)))
    build("too_far_back_first_block", far_first, lead=False)

    def far_later(d, lead_text, reach):
        d.dynamic(d.tokens_for(lead_text))
        t = recs(30)
        d.dynamic(_around(d, t, 10, (12, len(d.text) + 10 + reach)))
    build("too_far_back_later_block", lambda d: far_later(d, fastq(25, rng)[:4000].rsplit(b"\n@", 1)[0] + b"\n", 3000),
          lead=False)

    def far_handover(d):
        d.dynamic(d.tokens_for(fastq(3, rng)[:500].rsplit(b"\n@", 1)[0] + b"\n"))
        t = recs(15)
        d.dynamic(_around(d, t, 30, (10, 600)))
    build("too_far_back_after_handover", far_handover, lead=False)
    return out


REQUIRED_FEATURES = (
    {"stored", "fixed", "dynamic", "bfinal", "stored_pad_bits_set", "tiny_dynamic", "empty_dynamic"} |
    {"stored_%d_phase_%d" % (n, p) for n in (0, 65535) for p in range(8)} |
    {"lit_code_len_15", "dist_code_len_15", "rle_across_boundary", "cl16_6", "cl17_10", "cl18_138", "hclen_4",
     "hclen_19", "hlit_286", "hlit_trailing_zero", "hdist_trailing_zero", "len258_code284", "len258_code285",
     "dist_32768", "overlap_copy", "single_distance_code", "single_literal_code", "no_distance_codes", "too_far_back",
     "raw_symbol", "truncated"})


def test_legal_corpus_decodes_under_zlib():
    for c in legal_corpus():
        ok, got = zlib_verdict(c.deflate)
        assert ok, (c.name, got)
        assert got == c.text, c.name
        assert gzip.decompress(gzip_member(c.deflate, c.text)) == c.text


def bgzf_cases():
    return [c for c in legal_corpus() if 26 + len(c.deflate) <= 65536 and len(c.text) <= 65536]


def test_block_gzip_members_of_the_legal_corpus(lib, tmp_path):
    """The writer's block-gzip framing (the size in the "BC" subfield) through gzip and the host ingest path."""
    cases = bgzf_cases()
    assert len(cases) >= 5
    blob = b"".join(bgzf_member(c.deflate, c.text) for c in cases)
    assert gzip.decompress(blob) == b"".join(c.text for c in cases)
    pos = 0
    for c in cases:
        m = bgzf_member(c.deflate, c.text)
        assert blob[pos + 12:pos + 16] == b"BC\x02\x00" and struct.unpack_from("<H", blob, pos + 16)[0] == len(m) - 1
        pos += len(m)
    p = tmp_path / "corpus.bgzf.gz"
    p.write_bytes(blob)
    for threads in (1, 4):
        assert inflate(lib, p, threads, len(blob) * 4 + 65536) == normalised(b"".join(c.text for c in cases))


def test_invalid_corpus_is_rejected_by_zlib():
    for c in invalid_corpus():
        ok, why = zlib_verdict(c.deflate)
        assert not ok, c.name


def test_the_corpus_covers_every_feature():
    seen = set().union(*(c.features for c in legal_corpus() + invalid_corpus()))
    assert REQUIRED_FEATURES <= seen, sorted(REQUIRED_FEATURES - seen)
    # and the legal corpus alone carries every legal one
    legal = set().union(*(c.features for c in legal_corpus()))
    assert REQUIRED_FEATURES - {"hclen_4", "too_far_back", "raw_symbol", "truncated"} <= legal


def test_writer_codes_are_what_was_asked_for():
    from deflate_writer import limited_lengths
    rng = random.Random(5)
    for limit, n in ((7, 19), (9, 286), (12, 286), (15, 286)):
        freqs = [rng.choice([0, 1, 1, 2, 5, 1000, 1 << 20]) for _ in range(n)]
        lens = limited_lengths(freqs, limit)
        assert max(lens) <= limit and kraft(lens) == 1 << 15
        assert all((l > 0) == (f > 0) for l, f in zip(lens, freqs))


def member_file(tmp_path, c):
    blob = gzip_member(c.deflate, c.text) if "truncated" not in c.features else gzip_member(c.deflate, b"")[:-8]
    p = tmp_path / (c.name + ".gz")
    p.write_bytes(blob)
    return p


@pytest.fixture(scope="module")
def lib():
    from vfind_b200 import build
    build.build()
    from vfind_b200 import api
    L = api.load_library()
    L.vfb_debug_inflate_file.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_uint64,
                                         ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64),
                                         ctypes.POINTER(ctypes.c_uint64)]
    return L


# (threads, VFB_PGUNZIP_SEGMENT): 1 thread is the serial zlib path
HOST_PATHS = ((1, None), (2, 4096), (3, 9000), (4, 20000), (8, 4096), (5, 65536), (8, 400000), (6, None))


@pytest.mark.parametrize("name", [c.name for c in legal_corpus()])
def test_legal_streams_on_the_host_paths(lib, tmp_path, name):
    c = next(c for c in legal_corpus() if c.name == name)
    p = member_file(tmp_path, c)
    want = normalised(zlib_verdict(c.deflate)[1])
    for threads, segment in HOST_PATHS:
        assert inflate(lib, p, threads, len(c.text) + 64, segment) == want, (name, threads, segment)


@pytest.mark.parametrize("name", [c.name for c in invalid_corpus()])
def test_invalid_streams_fail_on_the_host_paths(lib, tmp_path, name):
    c = next(c for c in invalid_corpus() if c.name == name)
    assert c.text.count(b"\n") % 4 == 0          # FASTQ-shaped: only the deflate rule under test can fail
    p = member_file(tmp_path, c)
    for threads, segment in HOST_PATHS:
        with pytest.raises(RuntimeError):
            inflate(lib, p, threads, len(c.text) + 4096, segment)
            pytest.fail("%s decoded with %d threads, segment %s" % (name, threads, segment))
