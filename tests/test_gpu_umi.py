"""umi_length on the GPU against the reference (tests/umi_oracle.py)."""
import os
import random

import numpy as np
import pytest

import oracle
import strand_oracle
import umi_oracle
from conftest import write_fastq_gz
from vfind_b200 import api, find_variants

pytestmark = pytest.mark.gpu

PREFIX = b"GGGCCCAGCCGGCCGGAT"
SUFFIX = b"CCGGAGGCGGAGGTTCAG"
CODONS = [a + b + c for a in "ACGT" for b in "ACGT" for c in "ACGT" if a + b + c not in ("TAA", "TAG", "TGA")]


def molecule_reads(seed, n_mol, umi_len, umi_off, aa=(5, 40), both=False):
    """Reads drawn from a pool of molecules: each molecule (a UMI at umi_off, a variant from a small library) is read
    1-8 times, some copies with a substitution in the region; random tails make some reads too short for a UMI that
    reaches past the adapters; with `both` a third of the reads are reverse complements."""
    rng = random.Random(seed)
    lib = ["".join(rng.choice(CODONS) for _ in range(rng.randint(*aa))).encode() for _ in range(60)]
    umis = [bytes(rng.choice(b"ACGTN") for _ in range(umi_len)) for _ in range(max(1, n_mol // 3))]
    seqs = []
    for _ in range(n_mol):
        umi, region = rng.choice(umis), rng.choice(lib)
        lead = bytes(rng.choice(b"ACGT") for _ in range(umi_off)) + umi
        for _ in range(rng.randint(1, 8)):
            r = bytearray(region)
            if rng.random() < 0.15:
                r[rng.randrange(len(r))] = rng.choice(b"ACGTn")
            s = lead + PREFIX + bytes(r) + SUFFIX + bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 40)))
            if both and rng.random() < 0.33:
                s = strand_oracle.revcomp(s)
            seqs.append(s)
    rng.shuffle(seqs)
    return seqs


def spans_of(off, ln):
    s = np.zeros(len(off), dtype=api.SPAN_DTYPE)
    s["off"], s["len"] = off, ln
    return s


def rows_of(offsets, data, counts, mol):
    raw = data.tobytes()
    return {raw[int(offsets[i]):int(offsets[i + 1])]: (int(counts[i]), int(mol[i])) for i in range(len(counts))}


def gpu_table(seqs, umi_len, umi_off, skip_translation=False, batches=(), **kw):
    """One context; `batches`: the reads go in as consecutive submits of these sizes (the rest in one)."""
    text, off, ln = oracle.pack_reads(seqs)
    with api.Context((PREFIX, SUFFIX), device=0, skip_translation=skip_translation, umi_length=umi_len,
                     umi_offset=umi_off, **kw) as ctx:
        lo = 0
        for b in list(batches) + [len(seqs)]:
            hi = min(lo + b, len(seqs))
            if hi > lo:
                ctx.submit_host(text, spans_of(off[lo:hi], ln[lo:hi]))
            lo = hi
        o, d, c = ctx.finish_arrays()
        got = rows_of(o, d, c, ctx.molecules())
        info = ctx.umi_info()
        st = ctx.stats()
    return got, info, st


def oracle_table(seqs, umi_len, umi_off, skip_translation=False, both=False):
    return umi_oracle.umi_reads(seqs, oracle.make_params((PREFIX, SUFFIX), skip_translation=skip_translation), umi_len,
                                umi_off, both_strands=both)


# (skip_translation, umi_length, umi_offset, amino acids per region): UMIs across 4- and 16-byte word boundaries;
# composite keys of 60 aa + 16 (76 bytes) and 60 aa + 24 (84) sit on both sides of the fused kernel's 80-byte compare
CASES = [(False, 10, 0, (5, 40)), (True, 10, 0, (5, 20)), (False, 1, 3, (5, 40)), (False, 64, 5, (5, 40)),
         (True, 7, 13, (4, 12)), (False, 16, 1, (60, 60)), (False, 24, 2, (60, 60)), (True, 33, 30, (3, 9)),
         (False, 12, 80, (5, 20))]


@pytest.mark.parametrize("skip,k,o,aa", CASES)
def test_matches_oracle(skip, k, o, aa):
    # offset 80: a UMI past the adapters (the reads' own UMIs sit at 0), which the random tails leave short in some reads
    seqs = molecule_reads(k * 100 + o, 1500, k, o if o < 80 else 0, aa)
    want, short, pairs = oracle_table(seqs, k, o, skip)
    # first batch after a clear: k3_keys_tile + k4_insert; the next ones: k34_keys_count
    for batches in ((len(seqs),), (97,) * 6, (1000,)):
        got, info, st = gpu_table(seqs, k, o, skip, batches=batches)
        assert got == want
        assert info["pairs"] == pairs and info["rows_out"] == len(want) and info["reads_short"] == short
        # one submit: the key tile kernel only; several: the fused kernel's UMI instantiation ran too
        assert (st["fused_batches"] > 0) == (len(batches) > 1 or len(seqs) > batches[0])
    if o == 80:
        assert 0 < short < len(seqs)


def test_matches_oracle_without_the_fused_kernel():
    seqs = molecule_reads(5, 1500, 10, 2)
    want = oracle_table(seqs, 10, 2)[0]
    os.environ["VFB_FUSED_COUNT"] = "0"
    try:
        for skip in (False, True):
            got, _, st = gpu_table(seqs, 10, 2, skip, batches=(97,) * 5)
            assert got == oracle_table(seqs, 10, 2, skip)[0]
            assert st["fused_batches"] == 0
    finally:
        os.environ.pop("VFB_FUSED_COUNT", None)
    assert want


def test_one_bit_hash_decides_on_bytes():
    seqs = molecule_reads(9, 2000, 8, 0)
    want = oracle_table(seqs, 8, 0)[0]
    for batches in ((len(seqs),), (1000,)):
        got, _, _ = gpu_table(seqs, 8, 0, batches=batches, debug_hash_bits=1)
        assert got == want


def test_same_reads_twice_double_counts_not_molecules():
    seqs = molecule_reads(11, 1000, 10, 0)
    want = oracle_table(seqs, 10, 0)[0]
    got, info, _ = gpu_table(seqs + seqs, 10, 0, batches=(len(seqs),))
    assert got == {k: (2 * c, m) for k, (c, m) in want.items()}
    assert info["pairs"] == oracle_table(seqs, 10, 0)[2]


def test_finish_twice_and_resubmit():
    seqs = molecule_reads(12, 1000, 6, 4)
    text, off, ln = oracle.pack_reads(seqs)
    half = len(seqs) // 2
    with api.Context((PREFIX, SUFFIX), device=0, umi_length=6, umi_offset=4) as ctx:
        ctx.submit_host(text, spans_of(off[:half], ln[:half]))
        first = rows_of(*ctx.finish_arrays(), ctx.molecules())
        assert first == oracle_table(seqs[:half], 6, 4)[0]
        assert rows_of(*ctx.finish_arrays(), ctx.molecules()) == first
        with pytest.raises(RuntimeError):
            api._check(api.load_library().vfb_set_umi(ctx._h, 0, 8))     # the table is not empty
        ctx.submit_host(text, spans_of(off[half:], ln[half:]))
        assert rows_of(*ctx.finish_arrays(), ctx.molecules()) == oracle_table(seqs, 6, 4)[0]
        batch = ctx.finish_arrow()
        assert batch.schema.names == ["sequence", "count", "molecules"]
        got = {s.encode(): (c, m) for s, c, m in zip(*(batch.column(i).to_pylist() for i in range(3)))}
        assert got == oracle_table(seqs, 6, 4)[0]
        ctx.finish_arrays()                                  # the context holds a molecules column again
        ctx.table_clear()
        ctx.finish_arrays()                                  # an empty table: the info describes this finish
        info = ctx.umi_info()
        assert info["pairs"] == 0 and info["rows_out"] == 0 and info["ms"] == 0
        ctx.reset()
        api._check(api.load_library().vfb_set_umi(ctx._h, 0, 0))         # empty again: UMIs off
        ctx.submit_host(text, spans_of(off, ln))
        plain = oracle.process_reads(oracle.make_params((PREFIX, SUFFIX)), text, off, ln)[0]
        assert ctx.finish_dict() == plain
        with pytest.raises(RuntimeError):
            ctx.molecules()
        batch = ctx.finish_arrow()                           # no stale molecules column once UMIs are off
        assert batch.schema.names == ["sequence", "count"]
        assert {s.encode(): c for s, c in zip(batch.column(0).to_pylist(), batch.column(1).to_pylist())} == plain


@pytest.mark.parametrize("skip", [False, True])
def test_both_strands(skip):
    seqs = molecule_reads(13, 1500, 10, 0, both=True)
    want, short, _ = oracle_table(seqs, 10, 0, skip, both=True)
    got, info, st = gpu_table(seqs, 10, 0, skip, batches=(700,), both_strands=True)
    assert got == want and info["reads_short"] == short
    assert st["reverse_counted"] > 0


def test_two_contexts_merged_on_one_device(tmp_path):
    seqs = molecule_reads(14, 3000, 10, 0)
    want = oracle_table(seqs, 10, 0)[0]
    text, off, ln = oracle.pack_reads(seqs)
    half = len(seqs) // 2
    devs = [0, 1] if api._visible_devices() >= 2 else [0, 0]
    os.environ["VFB_MULTI_ALLOW_DUP"] = "1"
    try:
        with api.MultiContext((PREFIX, SUFFIX), devices=devs, umi_length=10) as m:
            m.contexts[0].submit_host(text, spans_of(off[:half], ln[:half]))
            m.contexts[1].submit_host(text, spans_of(off[half:], ln[half:]))
            o, d, c = m.finish_arrays()
            assert rows_of(o, d, c, m.molecules()) == want
            info = m.umi_info()
            assert info["rows_out"] == len(want)
        path = write_fastq_gz(tmp_path / "m.fq.gz", [("r%d" % i, s.decode(), "F" * len(s)) for i, s in enumerate(seqs)])
        frame = find_variants(path, (PREFIX.decode(), SUFFIX.decode()), show_progress=False, devices=devs, umi_length=10)
        cols = frame.to_pydict() if hasattr(frame, "to_pydict") else frame.to_dict(as_series=False)
        assert {s.encode(): (c, mo) for s, c, mo in zip(cols["sequence"], cols["count"], cols["molecules"])} == want
    finally:
        os.environ.pop("VFB_MULTI_ALLOW_DUP", None)


def test_partition_clear_absorb():
    torch = pytest.importorskip("torch")
    seqs = molecule_reads(15, 2000, 9, 1)
    want = oracle_table(seqs, 9, 1)[0]
    text, off, ln = oracle.pack_reads(seqs)
    with api.Context((PREFIX, SUFFIX), device=0, umi_length=9, umi_offset=1) as src:
        src.submit_host(text, spans_of(off, ln))
        for n_parts in (2, 3):
            sizes = src.partition_sizes(n_parts)
            offs = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64)
            buf = torch.empty(int(sum(sizes)), dtype=torch.uint8, device="cuda")
            src.partition_fill(n_parts, buf.data_ptr(), offs)
            merged = {}
            for p in range(n_parts):
                with api.Context((PREFIX, SUFFIX), device=0, umi_length=9, umi_offset=1) as dst:
                    dst.absorb(buf.data_ptr() + int(offs[p]), sizes[p])
                    part = rows_of(*dst.finish_arrays(), dst.molecules())
                assert not (set(part) & set(merged))          # every variant lands on one part with all its UMIs
                merged.update(part)
            assert merged == want
            torch.cuda.synchronize()


@pytest.mark.parametrize("members", [1, 40])
def test_find_variants_on_gzip_files(tmp_path, members):
    seqs = molecule_reads(16, 2000, 12, 3)
    want = oracle_table(seqs, 12, 3)[0]
    path = write_fastq_gz(tmp_path / "u.fq.gz", [("r%d" % i, s.decode(), "F" * len(s)) for i, s in enumerate(seqs)],
                          members=members)
    frame = find_variants(path, (PREFIX.decode(), SUFFIX.decode()), show_progress=False, device=0, umi_length=12,
                          umi_offset=3)
    cols = frame.to_pydict() if hasattr(frame, "to_pydict") else frame.to_dict(as_series=False)
    assert list(cols) == ["sequence", "count", "molecules"]
    assert {s.encode(): (c, m) for s, c, m in zip(cols["sequence"], cols["count"], cols["molecules"])} == want
    plain = find_variants(path, (PREFIX.decode(), SUFFIX.decode()), show_progress=False, device=0)
    cols = plain.to_pydict() if hasattr(plain, "to_pydict") else plain.to_dict(as_series=False)
    assert list(cols) == ["sequence", "count"]


def test_read_diagnostics_umi_column():
    seqs = molecule_reads(17, 60, 8, 2, both=True)[:200] + [b"ACGT"]
    tbl = api.read_diagnostics(seqs, (PREFIX, SUFFIX), both_strands=True, umi_length=8, umi_offset=2)
    umi = tbl.column("umi").to_pylist()
    strand = tbl.column("strand").to_pylist()
    for s, u, st in zip(seqs, umi, strand):
        if st is None:
            assert u is None
        else:
            r = s if st == 1 else strand_oracle.revcomp(s)
            assert u == r[2:10]
    assert "umi" not in api.read_diagnostics(seqs[:5], (PREFIX, SUFFIX)).column_names
