"""collapse_ratio on the GPU against tests/collapse_oracle.py: the standalone collapse over random tables (every key
length around the 4-byte words of the hash, bytes 0x00 and 0xFF, counts past 2^32 and near 2^53, counts exactly at
ratio * count), independent of row order and of the hash width; and the collapse inside find_variants, Context and
MultiContext, against the reference applied to the oracle's table."""
import os
import random

import numpy as np
import pyarrow as pa
import pytest

import collapse_oracle as co
import oracle
import strand_oracle
from conftest import write_fastq_gz
from test_gpu_strands import make_reads as make_strand_reads
from vfind_b200 import api, find_variants

pytestmark = pytest.mark.gpu

LENGTHS = [1, 2, 3, 4, 5, 7, 8, 9, 12, 13, 16, 17, 31, 32, 33, 63, 64, 65, 79, 80, 81, 127, 128, 129, 198, 255, 256, 257, 300]
ALPHABETS = [b"ACGT", b"ACGTN", b"ACDEFGHIKLMNPQRSTVWY*X", bytes([0x00, 0xFF, 0x41, 0x80])]


def mutate(rng, key, alphabet):
    p = rng.randrange(len(key))
    x = rng.choice([b for b in alphabet if b != key[p]])
    return key[:p] + bytes([x]) + key[p + 1:]


def make_table(rng, L, alphabet, n_parents, scale=1):
    """Parents with error tails (stars and chains), tied and exactly-at-ratio counts, other lengths, zero counts."""
    t = {}
    for _ in range(n_parents):
        k = bytes(rng.choice(alphabet) for _ in range(L + rng.choice((0, 0, 0, 1))))
        c = rng.choice((1, 4, 10, 64, 1000, 2 ** 33 + 3, 2 ** 53 - 1, 2 ** 53 + 2)) * scale
        t[k] = c
        cur = k
        for _ in range(rng.randrange(0, 10)):
            base = cur if rng.random() < 0.4 else k
            m = mutate(rng, base, alphabet)
            if m in t:
                continue
            cb = t[base]
            t[m] = max(1, rng.choice((1, 2, 3, cb, cb // 2, cb // 2 + 1, cb // 10, (cb + 1) // 2)))
            cur = m
    for k in list(t)[:2]:
        if rng.random() < 0.3:
            t[k] = 0
    return t


def to_table(d, rng=None, string=False):
    items = list(d.items())
    if rng is not None:
        rng.shuffle(items)
    typ = pa.string() if string else pa.binary()
    seq = [k.decode() if string else k for k, _ in items]
    return pa.table({"sequence": pa.array(seq, type=typ), "count": pa.array([v for _, v in items], type=pa.uint64())})


def as_dict(tbl):
    cols = tbl.to_pydict() if hasattr(tbl, "to_pydict") else tbl.to_dict(as_series=False)
    out = {}
    for k, v in zip(cols["sequence"], cols["count"]):
        k = k.encode() if isinstance(k, str) else k
        assert k not in out
        out[k] = v
    return out


def gpu_collapse(d, ratio, rng=None, **kw):
    return as_dict(api.collapse_variants(to_table(d, rng), ratio, **kw))


@pytest.mark.parametrize("alphabet", ALPHABETS, ids=["dna", "dna_n", "protein", "bytes"])
def test_standalone_matches_reference(alphabet):
    rng = random.Random(sum(alphabet))
    for L in LENGTHS:
        t = {}
        for _ in range(3):
            t.update(make_table(rng, L, alphabet, rng.randrange(2, 8)))
        # some rows of neighbouring lengths in the same call
        t.update(make_table(rng, max(1, L - 1), alphabet, 2))
        for ratio in (1, 1.5, 2, 10, 1e300):
            want = co.collapse_reference(t, ratio)
            assert gpu_collapse(t, ratio) == want, (L, ratio)
        want = co.collapse_reference(t, 2)
        assert gpu_collapse(t, 2, rng) == want                       # rows shuffled
        assert gpu_collapse(t, 2, rng, debug_hash_bits=8) == want, L
        # a 1- or 2-bit hash puts every pair into one probe run: a smaller table keeps that quadratic walk short
        small = make_table(rng, L, alphabet, 2)
        want = co.collapse_reference(small, 1.5)
        for bits in (1, 2):
            assert gpu_collapse(small, 1.5, rng, debug_hash_bits=bits) == want, (L, bits)


def test_standalone_many_rows():
    rng = random.Random(4)
    t = {}
    for _ in range(4000):
        t.update(make_table(rng, 30, b"ACGT", 1))
    for ratio in (1, 2, 5):
        assert gpu_collapse(t, ratio, rng) == co.collapse_reference(t, ratio)


def test_standalone_edge_cases():
    assert gpu_collapse({}, 2) == {}
    assert gpu_collapse({b"ACGT": 7}, 2) == {b"ACGT": 7}
    assert gpu_collapse({b"ACGT": 0, b"ACGA": 3, b"": 2}, 1) == {b"ACGA": 3, b"": 2}
    assert gpu_collapse({b"A": 0}, 1) == {}
    with pytest.raises(ValueError):
        api.collapse_variants(pa.table({"sequence": [b"ACGT", b"ACGA", b"ACGT"], "count": pa.array([3, 1, 2], pa.uint64())}), 2)
    with pytest.raises(ValueError):
        api.collapse_variants(pa.table({"sequence": [b"AC"], "count": pa.array([2 ** 56], pa.uint64())}), 2)
    # a string column stays a string column; a RecordBatch and a sliced table are taken as well
    out = api.collapse_variants(to_table({b"AAAA": 10, b"AAAC": 1}, string=True), 2)
    assert pa.types.is_large_string(out.schema.field("sequence").type) and as_dict(out) == {b"AAAA": 11}
    tbl = to_table({b"AAAA": 10, b"AAAC": 1, b"CCCC": 5, b"CCCA": 2})
    assert as_dict(api.collapse_variants(tbl.to_batches()[0], 2)) == {b"AAAA": 11, b"CCCC": 7}
    assert as_dict(api.collapse_variants(tbl.slice(2), 2)) == {b"CCCC": 7}


def test_standalone_rejects_duplicates_whoever_claims_the_slot():
    """A duplicate key is rejected even when every group it belongs to is represented by a third key: each position of
    the duplicated key has a neighbour that differs there, and the rows come in every order."""
    rng = random.Random(12)
    cases = [[b"A", b"A", b"C"]]
    for L in (1, 2, 3, 5, 9):
        k = bytes(rng.choice(b"ACGT") for _ in range(L))
        cases.append([k, k] + [k[:p] + bytes([k[p] ^ 2]) + k[p + 1:] for p in range(L)])
    for keys in cases:
        for trial in range(12):
            order = list(range(len(keys)))
            rng.shuffle(order)
            tbl = pa.table({"sequence": pa.array([keys[i] for i in order], pa.binary()),
                            "count": pa.array([3 if i == 0 else 2 if i == 1 else 1 for i in order], pa.uint64())})
            for bits in (0, 1, 8):
                with pytest.raises(ValueError, match="same key twice"):
                    api.collapse_variants(tbl, 2, debug_hash_bits=bits)


def test_polars_frame_round_trip(tmp_path):
    """The frame find_variants returns (polars when installed) goes straight back into collapse_variants."""
    pl = pytest.importorskip("polars")
    cfg = noisy_cfg(False)
    path = str(tmp_path / "noisy.fq.gz")
    oracle.write_fastq(cfg, 0, 20000, path, bgzf=True)
    ad = tuple(a.decode() for a in oracle.synth_adapters(cfg))
    frame = find_variants(path, ad, show_progress=False, device=0)
    assert isinstance(frame, pl.DataFrame)
    out = api.collapse_variants(frame, 2)
    assert isinstance(out, pl.DataFrame)
    assert as_dict(out) == co.collapse_reference(as_dict(frame), 2)


def noisy_cfg(skip_translation):
    # a small library with heavy per-base noise inside the region: error tails around every member
    return oracle.synth_cfg(seed=77, read_len=120, adapter_len=20, region_len=45, n_variants=300, p_err=0.2, indel=0.5,
                            force_indel=0, frameshift=0.0, noise=0.01, n_rate=0.001)


@pytest.mark.parametrize("skip_translation", [False, True])
def test_find_variants_with_region_noise(tmp_path, skip_translation):
    cfg = noisy_cfg(skip_translation)
    path = str(tmp_path / "noisy.fq.gz")
    oracle.write_fastq(cfg, 0, 60000, path, bgzf=True)
    ad = tuple(a.decode() for a in oracle.synth_adapters(cfg))
    base = oracle.find_variants_file(path, ad, n_threads=8, skip_translation=skip_translation)
    for ratio in (1, 2, 10):
        want = co.collapse_reference(base, ratio)
        assert len(want) < len(base)
        got = as_dict(find_variants(path, ad, skip_translation=skip_translation, show_progress=False, device=0,
                                    collapse_ratio=ratio))
        assert got == want
    # unset: the table is the uncollapsed one
    assert as_dict(find_variants(path, ad, skip_translation=skip_translation, show_progress=False, device=0)) == base


PREFIX = b"GGGCCCAGCCGGCCGGAT"
SUFFIX = b"CCGGAGGCGGAGGTTCAG"


@pytest.mark.parametrize("skip_translation", [False, True])
def test_find_variants_both_strands(tmp_path, skip_translation):
    rng = random.Random(31)
    seqs = make_strand_reads(rng, PREFIX, SUFFIX, 20000, lib=40)
    # sequencing errors inside the reads (regions included)
    seqs = [bytes(rng.choice(b"ACGT") if rng.random() < 0.004 else b for b in s) for s in seqs]
    path = write_fastq_gz(tmp_path / "both.fq.gz", [("r%d" % i, s.decode(), "F" * len(s)) for i, s in enumerate(seqs)])
    text, off, ln = oracle.pack_reads(seqs)
    p = oracle.make_params((PREFIX, SUFFIX), skip_translation=skip_translation)
    base = strand_oracle.process_reads_both_strands(p, text, off, ln, n_threads=8)[0]
    want = co.collapse_reference(base, 2)
    assert len(want) < len(base)
    got = as_dict(find_variants(path, (PREFIX.decode(), SUFFIX.decode()), skip_translation=skip_translation,
                                show_progress=False, device=0, both_strands=True, collapse_ratio=2))
    assert got == want


def spans_of(off, ln):
    s = np.zeros(len(off), dtype=api.SPAN_DTYPE)
    s["off"], s["len"] = off, ln
    return s


def reads_of(cfg, first, n):
    text, off, ln = oracle.synth_reads(cfg, first, n)
    return text, spans_of(off, ln)


def oracle_table(cfg, n, **kw):
    text, off, ln = oracle.synth_reads(cfg, 0, n)
    return oracle.process_reads(oracle.make_params(oracle.synth_adapters(cfg), **kw), text, off, ln, n_threads=8)[0]


def test_context_finish_twice_and_resubmit():
    cfg = noisy_cfg(False)
    ad = oracle.synth_adapters(cfg)
    half, full = oracle_table(cfg, 20000), oracle_table(cfg, 50000)
    with api.Context(ad, device=0, collapse_ratio=3, debug_hash_bits=8) as ctx:
        ctx.submit_host(*reads_of(cfg, 0, 20000))
        first = ctx.finish_dict()
        assert first == co.collapse_reference(half, 3)
        info = ctx.collapse_info()
        assert info["rows_in"] == len(half) and info["rows_out"] == len(first) and info["ms"] > 0
        assert ctx.finish_dict() == first                    # the count table keeps every key
        ctx.submit_host(*reads_of(cfg, 20000, 30000))
        assert ctx.finish_dict() == co.collapse_reference(full, 3)
        assert ctx.collapse_info()["rows_in"] == len(full)
        st = ctx.stats()
        assert st["unique"] == len(full)                     # rows of the table, not of the result
    with api.Context(ad, device=0) as ctx:
        ctx.submit_host(*reads_of(cfg, 0, 20000))
        assert ctx.finish_dict() == half
        assert ctx.collapse_info() == {"rows_in": 0, "rows_out": 0, "ms": 0.0}


def test_multi_context_two_contexts():
    if api._visible_devices() >= 2:
        devs = [0, 1]
    else:
        os.environ["VFB_MULTI_ALLOW_DUP"] = "1"
        devs = [0, 0]
    cfg = noisy_cfg(False)
    ad = oracle.synth_adapters(cfg)
    base = oracle_table(cfg, 40000)
    want = co.collapse_reference(base, 2)
    with api.MultiContext(ad, devices=devs, collapse_ratio=2) as m:
        m.contexts[0].submit_host(*reads_of(cfg, 0, 20000))
        m.contexts[1].submit_host(*reads_of(cfg, 20000, 20000))
        assert m.finish_dict() == want
        info = m.collapse_info()
        assert info["rows_in"] == len(base) and info["rows_out"] == len(want)
        batch = m.finish_arrow()
        assert {k.encode(): v for k, v in zip(batch.column(0).to_pylist(), batch.column(1).to_pylist())} == want
    with api.Context(ad, device=0, collapse_ratio=2) as ctx:
        ctx.submit_host(*reads_of(cfg, 0, 40000))
        assert ctx.finish_dict() == want
