"""The hand-built deflate corpus of test_deflate_streams_cpu.py through the device decoders: k_inflate_warp (block-gzip
members, vfb_debug_gpu_inflate) and the single-stream device gunzip (k_gz_* + gunzip_gpu.cu, vfb_debug_inflate_file with
VFB_GPU_GUNZIP=2).  Legal streams must decode to zlib's output, invalid ones must fail as zlib fails; then find_variants
on a block-gzip and a plain gzip file written by the same writer must equal the oracle's table."""
import os
import random

import pytest

from deflate_writer import Deflate, bgzf_member, gzip_member, zlib_verdict
from test_deflate_streams_cpu import invalid_corpus, legal_corpus, member_file
from test_gpu_gunzip import gpu_inflate as stream_inflate
from test_gpu_gunzip import lib  # noqa: F401  (fixture)
from test_gpu_inflate import gpu_inflate as member_inflate
from test_pgunzip_cpu import normalised

pytestmark = pytest.mark.gpu


def kernel_member(c):
    """A block-gzip member when the case fits one (64 KiB of member), else a plain gzip member: the kernel takes any
    member header, the size field only matters to the reader that splits a file into members."""
    if "truncated" in c.features:
        return gzip_member(c.deflate, b"")[:-8]
    if 26 + len(c.deflate) <= 65536 and len(c.text) <= 65536:
        return bgzf_member(c.deflate, c.text)
    return gzip_member(c.deflate, c.text)


def test_legal_corpus_on_the_block_gzip_kernel():
    cases = legal_corpus()
    want = [zlib_verdict(c.deflate)[1] for c in cases]
    got, bad, _ = member_inflate([kernel_member(c) for c in cases], [len(w) for w in want])
    assert bad == 0xFFFFFFFF
    assert got == b"".join(want)


@pytest.mark.parametrize("name", [c.name for c in invalid_corpus()])
def test_invalid_members_are_reported_by_the_block_gzip_kernel(name):
    c = next(c for c in invalid_corpus() if c.name == name)
    good = next(g for g in legal_corpus() if g.name == "one_code_and_no_codes")
    members = [kernel_member(good), kernel_member(c), kernel_member(good)]
    got, bad, _ = member_inflate(members, [len(good.text), len(c.text), len(good.text)])
    assert bad == 1, name
    assert got[:len(good.text)] == good.text and got[len(good.text) + len(c.text):] == good.text     # neighbours intact


# (VFB_GUNZIP_SEGMENT, VFB_GUNZIP_GAP, VFB_GUNZIP_CAP, VFB_GUNZIP_HOST_QUOTA): GAP = 64 makes nearly every block its own
# chunk (windows through chains of short chunks), small capacities hand chunks to zlib and a quota of 1 hands them back
STREAM_CONFIGS = ((None, None, None, None), (None, 64, None, None), (4096, 64, None, None), (65536, 64, 20000, 1),
                  (None, 512, 1024, 1), (300000, 64, 1024, None), (20000, 2048, 40000, 100000))


@pytest.mark.parametrize("name", [c.name for c in legal_corpus()])
def test_legal_streams_on_the_single_stream_device_decoder(lib, tmp_path, name):  # noqa: F811
    c = next(c for c in legal_corpus() if c.name == name)
    p = member_file(tmp_path, c)
    want = normalised(zlib_verdict(c.deflate)[1])
    for cfg in STREAM_CONFIGS:
        assert stream_inflate(lib, p, len(c.text) + 64, *cfg) == want, (name, cfg)


@pytest.mark.parametrize("name", [c.name for c in invalid_corpus()])
def test_invalid_streams_fail_on_the_single_stream_device_decoder(lib, tmp_path, name):  # noqa: F811
    c = next(c for c in invalid_corpus() if c.name == name)
    p = member_file(tmp_path, c)
    for cfg in STREAM_CONFIGS:
        with pytest.raises(RuntimeError):
            stream_inflate(lib, p, len(c.text) + 4096, *cfg)
            pytest.fail("%s decoded with %s" % (name, cfg))


def test_distance_before_the_stream_in_a_later_chunk(lib, tmp_path):  # noqa: F811
    """~4 KB of text, then a non-final dynamic block (a chunk of its own with GAP = 64) whose match reaches before the
    stream's first byte: the chunk after the first must be checked against the history that exists, not just chunk 0."""
    c = next(c for c in invalid_corpus() if c.name == "too_far_back_later_block")
    p = member_file(tmp_path, c)
    with pytest.raises(RuntimeError, match="too far back"):
        stream_inflate(lib, p, len(c.text) + 4096, None, 64)


def test_distance_before_the_stream_after_the_handover_to_zlib(lib, tmp_path):  # noqa: F811
    """~500 bytes of text, then a chunk larger than the chunk capacity (zlib takes it over with the text so far as its
    dictionary) reaching 600 bytes back: zlib must be given only the text that exists."""
    c = next(c for c in invalid_corpus() if c.name == "too_far_back_after_handover")
    p = member_file(tmp_path, c)
    with pytest.raises(RuntimeError, match="too far back"):
        stream_inflate(lib, p, len(c.text) + 4096, None, 64, 1024)


def _writer_stream(text, rng, final=True, d=None):
    """`text` as a mix of tiny and large dynamic blocks, fixed and stored blocks, some with 15-bit codes."""
    d = d or Deflate()
    pos = 0
    while pos < len(text):
        n = min(rng.choice([50, 300, 3000, 20000]), len(text) - pos)
        piece, last = text[pos:pos + n], final and pos + n >= len(text)
        k = rng.randrange(6)
        if k == 0 and n <= 65535:
            d.stored(piece, final=last)
        elif k == 1:
            d.fixed(d.tokens_for(piece), final=last)
        elif k == 2:
            d.dynamic(d.tokens_for(piece), final=last, lit_weights={0xC0 + j: 1 << (j + 3) for j in range(26)})
        else:
            d.dynamic(d.tokens_for(piece), final=last)
        pos += n
    return d


def test_find_variants_on_files_from_the_writer(tmp_path):
    import oracle
    from test_gpu_parity import PREFIX, SUFFIX, make_reads
    from vfind_b200 import find_variants
    rng = random.Random(1953)
    seqs = make_reads(rng, PREFIX, SUFFIX, 6000, lib=300)
    ad = (PREFIX.decode(), SUFFIX.decode())
    text = "".join("@r%d\n%s\n+\n%s\n" % (i, s.decode(), "F" * len(s)) for i, s in enumerate(seqs)).encode()
    # block gzip: members of at most ~60 KB of text cut at record boundaries, then the empty end-of-file member
    members, pos = [], 0
    while pos < len(text):
        end = len(text) if len(text) - pos <= 60000 else text.rfind(b"\n@", pos, pos + 60000) + 1
        d = _writer_stream(text[pos:end], rng)
        members.append(bgzf_member(d.getvalue(), d.text))
        pos = end
    e = Deflate()
    e.fixed([], final=True)
    bgzf = tmp_path / "writer.bgzf.fq.gz"
    bgzf.write_bytes(b"".join(members) + bgzf_member(e.getvalue(), b""))
    d = _writer_stream(text, rng)
    assert d.text == text
    plain = tmp_path / "writer.plain.fq.gz"
    plain.write_bytes(gzip_member(d.getvalue(), text))
    for p, env in ((bgzf, {}), (plain, {"VFB_GPU_GUNZIP": "2", "VFB_GUNZIP_GAP": "64"})):
        want = oracle.find_variants_file(str(p), (PREFIX, SUFFIX), n_threads=4)
        os.environ.update(env)
        try:
            out = find_variants(str(p), ad, n_threads=4, show_progress=False)
        finally:
            for k in env:
                os.environ.pop(k, None)
        cols = out.to_pydict() if hasattr(out, "to_pydict") else out.to_dict(as_series=False)
        assert {k.encode(): v for k, v in zip(cols["sequence"], cols["count"])} == want, p.name
