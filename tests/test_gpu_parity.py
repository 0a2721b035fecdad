"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle, bit for bit.

Every test here needs a B200 (`-m gpu`).  Per-read diagnostics (exact positions, integer
scores, alignment lengths, accept decisions, boundaries) and the final table must be
identical to the oracle's on the same inputs.
"""
import random

import numpy as np
import pytest

import oracle
from vfind_b200 import api

pytestmark = pytest.mark.gpu

PREFIX = b"GGGCCCAGCCGGCCGGAT"
SUFFIX = b"CCGGAGGCGGAGGTTCAG"


def spans_of(off, ln):
    s = np.zeros(len(off), dtype=api.SPAN_DTYPE)
    s["off"], s["len"] = off, ln
    return s


def gpu_run(seqs, adapters, want_diag=True, **kw):
    text, off, ln = oracle.pack_reads(seqs)
    with api.Context(adapters, diagnostics=want_diag, **kw) as ctx:
        ctx.submit_host(text, spans_of(off, ln))
        diag = ctx.diag(len(seqs)) if want_diag and len(seqs) else None
        table = ctx.finish_dict()
        stats = ctx.stats()
    return table, diag, stats


def oracle_run(seqs, adapters, **kw):
    text, off, ln = oracle.pack_reads(seqs)
    okw = {k: v for k, v in kw.items() if k in ("match_score", "mismatch_score", "gap_open_penalty",
                                                "gap_extend_penalty", "accept_prefix_alignment",
                                                "accept_suffix_alignment", "skip_translation")}
    p = oracle.make_params(adapters, **okw)
    return oracle.process_reads(p, text, off, ln, n_threads=4, want_diag=True)


def assert_diag_equal(got, want, compute_all=True):
    for f in ("exact_prefix", "exact_suffix", "score_prefix", "len_prefix", "start"):
        assert (got[f] == want[f]).all(), (f, np.nonzero(got[f] != want[f])[0][:5])
    if compute_all:
        for f in ("score_suffix", "len_suffix", "end"):
            assert (got[f] == want[f]).all(), (f, np.nonzero(got[f] != want[f])[0][:5])


def mutate(rng, ad, max_edits=3, alphabet=b"ACGT"):
    inst = bytearray(ad)
    for _ in range(rng.randrange(0, max_edits + 1)):
        if not inst:
            break
        k = rng.randrange(len(inst))
        op = rng.randrange(3)
        if op == 0:
            inst[k] = rng.choice(alphabet)
        elif op == 1:
            del inst[k]
        else:
            inst.insert(k, rng.choice(alphabet))
    return bytes(inst)


def make_reads(rng, pre, suf, n, var_lens=(21, 21, 24, 22, 30), lead=(0, 6), alphabet=b"ACGT", lib=24):
    # (regions are drawn from `alphabet` too: lower case, U, N and other bytes reach the translate kernel's tables)
    variants = [bytes(rng.choice(alphabet) for _ in range(rng.choice(var_lens))) for _ in range(lib)]
    seqs = []
    for _ in range(n):
        a = pre if rng.random() < 0.5 else mutate(rng, pre, alphabet=alphabet)
        b = suf if rng.random() < 0.5 else mutate(rng, suf, alphabet=alphabet)
        ld = bytes(rng.choice(alphabet) for _ in range(rng.randrange(lead[0], lead[1] + 1)))
        tl = bytes(rng.choice(alphabet) for _ in range(rng.randrange(lead[0], lead[1] + 1)))
        seqs.append(ld + a + rng.choice(variants) + b + tl)
    return seqs


def test_toy_file_end_to_end(toy_gz, golden):
    # tests/test_vfind.py:5-13 of the reference, through the drop-in function
    from vfind import find_variants
    toy = golden["toy"]
    out = find_variants(toy_gz, tuple(toy["adapters"]), show_progress=False)
    cols = out.to_pydict() if hasattr(out, "to_pydict") else out.to_dict(as_series=False)
    assert list(cols.keys()) == ["sequence", "count"]
    assert sorted(zip(cols["sequence"], cols["count"])) == sorted((k, v) for k, v in toy["table"])
    assert oracle.find_variants_file(toy_gz, toy["adapters"]) == {k.encode(): v for k, v in toy["table"]}


def test_toy_diag(golden):
    toy = golden["toy"]
    seqs = [r["seq"].encode() for r in toy["reads"]]
    ad = tuple(a.encode() for a in toy["adapters"])
    table, diag, stats = gpu_run(seqs, ad)
    otable, odiag, cells = oracle_run(seqs, ad)
    assert table == otable == {b"MAGICAL": 4}
    assert_diag_equal(diag, odiag)
    assert stats["dp_cells"] == cells and stats["dp_kernel_kind"] == 1
    assert stats["counted"] == 4 and stats["unique"] == 1 and stats["kernel_launches"] > 0


def test_unit_vectors(golden):
    # src/lib.rs:339-369 through the GPU DP
    for v in golden["unit_vectors"]:
        a, s = v["adapter"].encode(), v["seq"].encode()
        ad = (a, SUFFIX) if v["is_prefix"] else (PREFIX, a)
        _, diag, _ = gpu_run([s], ad)
        score = diag[0]["score_prefix" if v["is_prefix"] else "score_suffix"]
        assert (float(score) > 40.5) == v["accept"]
        assert score == oracle.sg_stats(a, s)[0]


def test_kats_rule_discriminating():
    # SURVEY §8(c): what the assumed parasail rules predict, on the GPU
    _, d, _ = gpu_run([b"TCTCCAGGTAAAGCGGGCTCAT"], (b"TCTCCAGGTAAG", SUFFIX))
    assert (d[0]["score_prefix"], d[0]["len_prefix"]) == (31, 12)
    _, d, _ = gpu_run([b"CTATATTGCGAGGCAACAGCAAGGAGA"], (b"CTTATATGCGAG", SUFFIX))
    assert (d[0]["score_prefix"], d[0]["len_prefix"]) == (23, 13)


@pytest.mark.parametrize("scoring", [(3, -2, 5, 2), (1, -1, 0, 0), (2, -3, 4, 1), (5, -4, 10, 1),
                                     (1, -1, 1, 1), (2, -1, 3, 0), (4, -6, 0, 3)])
@pytest.mark.parametrize("thr", [0.75, 0.6])
def test_random_parity_scoring(scoring, thr):
    rng = random.Random(hash((scoring, thr)) & 0xFFFF)
    seqs = make_reads(rng, PREFIX, SUFFIX, 1500)
    kw = dict(match_score=scoring[0], mismatch_score=scoring[1], gap_open_penalty=scoring[2],
              gap_extend_penalty=scoring[3], accept_prefix_alignment=thr, accept_suffix_alignment=thr)
    table, diag, stats = gpu_run(seqs, (PREFIX, SUFFIX), **kw)
    otable, odiag, cells = oracle_run(seqs, (PREFIX, SUFFIX), **kw)
    assert_diag_equal(diag, odiag)
    assert table == otable
    assert stats["dp_cells"] == cells


@pytest.mark.parametrize("A", [1, 2, 3, 4, 5, 7, 8, 9, 12, 17, 19, 20, 21, 31, 32, 33, 40, 47, 48, 57, 63, 64])
def test_random_parity_adapter_lengths(A):
    rng = random.Random(1000 + A)
    pre = bytes(rng.choice(b"ACGT") for _ in range(A))
    suf = bytes(rng.choice(b"ACGT") for _ in range(A))
    seqs = make_reads(rng, pre, suf, 600, lead=(0, 9))
    seqs += [b"A", b"AC", pre[: max(1, A - 1)], pre, suf, pre + suf, pre + b"ACG" + suf]
    table, diag, _ = gpu_run(seqs, (pre, suf), accept_prefix_alignment=0.6, accept_suffix_alignment=0.7)
    otable, odiag, _ = oracle_run(seqs, (pre, suf), accept_prefix_alignment=0.6, accept_suffix_alignment=0.7)
    assert_diag_equal(diag, odiag)
    assert table == otable


@pytest.mark.parametrize("A", [65, 100, 200])
def test_long_adapters_use_fallback_kernel(A):
    rng = random.Random(A)
    pre = bytes(rng.choice(b"ACGT") for _ in range(A))
    suf = bytes(rng.choice(b"ACGT") for _ in range(A))
    seqs = make_reads(rng, pre, suf, 200)
    table, diag, stats = gpu_run(seqs, (pre, suf))
    otable, odiag, _ = oracle_run(seqs, (pre, suf))
    assert stats["dp_kernel_kind"] == 2
    assert_diag_equal(diag, odiag)
    assert table == otable


def test_fallback_kernel_matches_packed_kernel():
    rng = random.Random(77)
    seqs = make_reads(rng, PREFIX, SUFFIX, 2000, alphabet=b"ACGTNacgtn")
    a = gpu_run(seqs, (PREFIX, SUFFIX))
    b = gpu_run(seqs, (PREFIX, SUFFIX), force_generic_dp=True)
    assert a[2]["dp_kernel_kind"] == 1 and b[2]["dp_kernel_kind"] == 2
    assert a[0] == b[0]
    assert_diag_equal(a[1], b[1])


def test_wildcards_case_and_u():
    # Q9: exact search is case-sensitive, the alignment matrix is case-insensitive and scores
    # non-ACGT as 0, translate maps U to T and anything else to X
    rng = random.Random(5)
    seqs = make_reads(rng, PREFIX, SUFFIX, 1500, alphabet=b"ACGTNacgtnUu-")
    seqs += [PREFIX.lower() + b"ATGAAA" + SUFFIX, PREFIX + b"AUGNNNUAA" + SUFFIX.lower(),
             PREFIX + b"atgcccggg" + SUFFIX]
    for skip in (False, True):
        table, diag, _ = gpu_run(seqs, (PREFIX, SUFFIX), skip_translation=skip)
        otable, odiag, _ = oracle_run(seqs, (PREFIX, SUFFIX), skip_translation=skip)
        assert_diag_equal(diag, odiag)
        assert table == otable


TRIPLET_ALPHABET = b"ACGTUacgtuN-"


@pytest.mark.parametrize("skip", [False, True])
@pytest.mark.parametrize("windowed", [False, True])
def test_translate_all_triplets(skip, windowed):
    """Every triplet over the 10 accepted letters x 3 positions of ASCII_TO_INDEX (src/lib.rs:86-95) plus 'N', '-'
    and a non-ASCII byte reaches k3_keys_tile's three premultiplied LUTs and the codon table (src/lib.rs:16-44,
    :52-77): once as a one-codon region, and in 7-codon regions at every codon position; with skip_translation
    the raw regions (valid and invalid UTF-8) are the keys (src/lib.rs:294-297)."""
    letters = list(TRIPLET_ALPHABET) + [0xC3]
    triplets = [bytes((a, b, c)) for a in letters for b in letters for c in letters]
    assert len(triplets) == 13 ** 3
    rng = random.Random(17)
    seqs = [PREFIX + t + SUFFIX for t in triplets]
    order = triplets[:]
    for rot in range(7):                       # every triplet at each of the 7 codon positions of a region
        rng.shuffle(order)
        for i in range(0, len(order) - 6, 7):
            grp = order[i:i + 7]
            seqs.append(PREFIX + b"".join(grp[rot:] + grp[:rot]) + SUFFIX)
    seqs += [PREFIX + t + b"\xa9" + b"ACG" + SUFFIX for t in triplets[:300]]     # 7-byte regions: partial codon / UTF-8 pairs
    if windowed:
        text, off, ln = oracle.pack_reads(seqs)
        with api.Context((PREFIX, SUFFIX), skip_translation=skip) as ctx:
            ctx.submit_host(text, spans_of(off, ln))
            table = ctx.finish_dict()
            assert ctx.stats()["dp_kernel_kind"] == 3
    else:
        table, _, _ = gpu_run(seqs, (PREFIX, SUFFIX), skip_translation=skip)
    otable, _, _ = oracle_run(seqs, (PREFIX, SUFFIX), skip_translation=skip)
    assert table == otable
    if not skip:
        # the oracle's own table is the reference's AA_TABLE_CANONICAL (pinned by tests/golden): spot checks
        assert otable[b"M"] >= 1 and otable[b"*"] >= 3 and b"X" in otable
        assert sum(otable.values()) >= 13 ** 3


def test_adapter_with_wildcard_bases():
    rng = random.Random(6)
    pre, suf = b"GGGCCNAGCCGGCCGGAT", b"CCGGAGGCGGaGGTTCAG"
    seqs = make_reads(rng, pre, suf, 800, alphabet=b"ACGTN")
    table, diag, _ = gpu_run(seqs, (pre, suf))
    otable, odiag, _ = oracle_run(seqs, (pre, suf))
    assert_diag_equal(diag, odiag)
    assert table == otable


@pytest.mark.parametrize("pre,suf", [
    (b"ACACACACACACACACACAC", b"GTGTGTGTGTGTGTGTGTGT"),      # one 4-mer at every offset
    (b"AAAAAAAAAAAAAAAAAAAAAAAA", b"CCCCCCCCCCC"),            # homopolymers, stride 4 and 2
    (b"ACGTACGT", b"TTGACCA"),                                # stride 1
    (b"GGGCCCAGCCGGCCGGAT", b"GGGCCCAGCCGGCCGGATC"),          # one adapter contains the other
])
def test_scan_repetitive_and_nested_adapters(pre, suf):
    rng = random.Random(len(pre) * 131 + len(suf))
    seqs = []
    for _ in range(1500):
        parts = []
        for _ in range(rng.randrange(1, 6)):
            k = rng.randrange(5)
            if k == 0:
                parts.append(pre)
            elif k == 1:
                parts.append(suf)
            elif k == 2:
                parts.append(pre[:rng.randrange(len(pre))])
            elif k == 3:
                parts.append(bytes(rng.choice(pre + suf) for _ in range(rng.randrange(1, 30))))
            else:
                parts.append(bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(1, 40))))
        seqs.append(b"".join(parts))
    kw = dict(accept_prefix_alignment=1.0, accept_suffix_alignment=1.0, skip_translation=True)
    fast = gpu_run(seqs, (pre, suf), **kw)
    slow = gpu_run(seqs, (pre, suf), force_general_scan=True, **kw)
    otable, odiag, _ = oracle_run(seqs, (pre, suf), **kw)
    assert_diag_equal(fast[1], odiag)
    assert_diag_equal(slow[1], odiag)
    assert fast[0] == slow[0] == otable


def _scan_only(text, off, ln, adapters, **kw):
    kw = dict(accept_prefix_alignment=1.0, accept_suffix_alignment=1.0, skip_translation=True, **kw)
    with api.Context(adapters, diagnostics=True, **kw) as ctx:
        ctx.submit_host(text, spans_of(off, ln))
        diag = ctx.diag(len(off))
        table = ctx.finish_dict()
    return table, diag


@pytest.mark.parametrize("pre,suf", [
    (b"GGGCCCAGCCGGCCGGATTA", b"CCGGAGGCGGAGGTTCAGAC"),                      # 8-byte keys every 8 bytes
    (b"GGGCCCAGCCGGCCGGATTACGATCGGA", b"CCGGAGGCGGAGGTTCAGACTTGACCATGCAAT"),    # 8-byte keys every 16 bytes
])
def test_scan_tile_candidates_and_scattered_spans(pre, suf):
    """The tile scan (kernels_scan.cu, k1_scan_tile): decoy keys that fail verification before a real
    occurrence, repeated adapters (leftmost wins, src/lib.rs:148), occurrences cut by a read end or
    continued in the next read, empty / short / very long reads, and span orders that make a warp's
    text range exceed its tile (byte-wise path) -- against the oracle and the byte-wise kernel."""
    rng = random.Random(len(pre) * 7 + 3)
    rnd = lambda n: bytes(rng.choice(b"ACGT") for _ in range(n))
    seqs = []
    for i in range(6000):
        k = rng.randrange(12)
        if k == 0:      # decoy (adapter head, then a mismatch) before the real thing
            seqs.append(rnd(rng.randrange(0, 9)) + pre[:rng.randrange(8, len(pre))] + b"N" + rnd(rng.randrange(0, 20)) + pre +
                        rnd(30) + suf[:rng.randrange(8, len(suf))] + rnd(3) + suf + rnd(rng.randrange(0, 9)))
        elif k == 1:    # adapters twice
            seqs.append(rnd(rng.randrange(0, 17)) + pre + rnd(rng.randrange(0, 40)) + pre + rnd(21) + suf + rnd(rng.randrange(0, 40)) + suf)
        elif k == 2:    # occurrence cut by the read end; the rest opens the next read
            cut = rng.randrange(1, len(pre))
            seqs.append(rnd(rng.randrange(0, 60)) + pre[:cut])
            seqs.append(pre[cut:] + rnd(rng.randrange(0, 60)) + suf[:rng.randrange(1, len(suf))])
        elif k == 3:
            seqs.append(b"" if rng.random() < 0.5 else rnd(rng.randrange(1, len(pre))))
        elif k == 4 and i % 50 == 0:
            seqs.append(rnd(rng.randrange(3000, 9000)) + pre + rnd(300) + suf + rnd(rng.randrange(0, 3000)))
        elif k == 5:    # suffix before prefix, overlapping adapters
            seqs.append(suf + pre[:5] + pre + rnd(12))
        else:
            seqs.append(rnd(rng.randrange(0, 13)) + pre + rnd(rng.choice((21, 24, 30, 198))) + suf + rnd(rng.randrange(0, 13)))
    text, off, ln = oracle.pack_reads(seqs)
    want, odiag, _ = oracle.process_reads(oracle.make_params((pre, suf), accept_prefix_alignment=1.0, accept_suffix_alignment=1.0,
                                                             skip_translation=True), text, off, ln, want_diag=True)
    got, diag = _scan_only(text, off, ln, (pre, suf))
    assert_diag_equal(diag, odiag)
    assert got == want
    slow, sdiag = _scan_only(text, off, ln, (pre, suf), force_general_scan=True)
    assert_diag_equal(sdiag, odiag)
    # the same reads visited in a random order (a warp's 32 reads span the whole buffer), and in an
    # order that is sorted except for every 7th read
    n = len(off)
    swapped = np.arange(n)
    for i in range(0, n // 2, 7):
        swapped[i], swapped[n - 1 - i] = n - 1 - i, i
    for order in (np.array(rng.sample(range(n), n)), swapped):
        got2, diag2 = _scan_only(text, off[order], ln[order], (pre, suf))
        for f in ("exact_prefix", "exact_suffix", "start", "end"):
            assert (diag2[f] == odiag[f][order]).all(), f
        assert got2 == want


@pytest.mark.parametrize("skip_translation,region", [(True, 198), (False, 600), (False, 198)])
def test_key_blocks_larger_than_the_staging(skip_translation, region):
    """k3_keys_tile assembles a warp's keys in 4 KB of shared memory; 32 keys of 198 raw bytes (skip_translation)
    or 200 amino acids do not fit and are written to the arena directly -- same table either way."""
    rng = random.Random(region + int(skip_translation))
    rnd = lambda n: bytes(rng.choice(b"ACGT") for _ in range(n))
    lib = [rnd(region) for _ in range(40)]
    seqs = [rnd(rng.randrange(0, 5)) + PREFIX + rng.choice(lib) + SUFFIX + rnd(rng.randrange(0, 5)) for _ in range(3000)]
    kw = dict(skip_translation=skip_translation)
    got, diag, _ = gpu_run(seqs, (PREFIX, SUFFIX), **kw)
    want, odiag, _ = oracle_run(seqs, (PREFIX, SUFFIX), **kw)
    assert_diag_equal(diag, odiag)
    assert got == want and sum(want.values()) == 3000


def test_scan_unaligned_text_offsets():
    # reads at every byte alignment inside a larger text buffer (as FASTQ text delivers them)
    rng = random.Random(21)
    chunks, off, ln, pos = [], [], [], 0
    for i in range(3000):
        junk = bytes(rng.choice(b"@+FFFFF:#rs0123456789\n") for _ in range(rng.randrange(0, 23)))
        read = make_reads(rng, PREFIX, SUFFIX, 1)[0]
        chunks += [junk, read]
        off.append(pos + len(junk))
        ln.append(len(read))
        pos += len(junk) + len(read)
    text = np.frombuffer(b"".join(chunks), dtype=np.uint8)
    off, ln = np.array(off, np.uint32), np.array(ln, np.uint32)
    with api.Context((PREFIX, SUFFIX), diagnostics=True) as ctx:
        ctx.submit_host(text, spans_of(off, ln))
        diag = ctx.diag(len(off))
        got = ctx.finish_dict()
    want, odiag, _ = oracle.process_reads(oracle.make_params((PREFIX, SUFFIX)), text, off, ln, want_diag=True)
    assert_diag_equal(diag, odiag)
    assert got == want


def test_submit_device_unaligned_buffer():
    # a caller's device buffer whose ends are not 16-byte aligned: the library must not read
    # outside it (it runs on an aligned copy) and results must not change
    torch = pytest.importorskip("torch")
    rng = random.Random(22)
    seqs = make_reads(rng, PREFIX, SUFFIX, 4000)
    text, off, ln = oracle.pack_reads(seqs)
    want, odiag, _ = oracle_run(seqs, (PREFIX, SUFFIX))
    for shift in (0, 1, 3, 7, 13):
        big = torch.full((len(text) + 64,), ord("G"), dtype=torch.uint8, device="cuda")
        big[shift:shift + len(text)] = torch.from_numpy(text.copy()).cuda()
        sp = torch.from_numpy(np.stack([off, ln], 1).astype(np.uint32).view(np.int32).copy()).cuda()
        with api.Context((PREFIX, SUFFIX), diagnostics=True) as ctx:
            ctx.submit_device(big.data_ptr() + shift, len(text), sp.data_ptr(), len(seqs))
            diag = ctx.diag(len(seqs))
            got = ctx.finish_dict()
        assert_diag_equal(diag, odiag)
        assert got == want


def test_threshold_one_disables_alignment():
    rng = random.Random(8)
    seqs = make_reads(rng, PREFIX, SUFFIX, 800)
    for tp, ts in ((1.0, 0.75), (0.75, 1.0), (1.0, 1.0)):
        table, diag, stats = gpu_run(seqs, (PREFIX, SUFFIX), accept_prefix_alignment=tp, accept_suffix_alignment=ts)
        otable, odiag, cells = oracle_run(seqs, (PREFIX, SUFFIX), accept_prefix_alignment=tp, accept_suffix_alignment=ts)
        assert_diag_equal(diag, odiag)
        assert table == otable and stats["dp_cells"] == cells
        if tp == ts == 1.0:
            assert stats["dp_cells"] == 0


def test_float_threshold_edges():
    # Q3: 0.7*3*20 = 41.99999999999999 accepts 42; 0.8*3*20 = 48.00000000000001 rejects 48
    rng = random.Random(9)
    pre = bytes(rng.choice(b"ACGT") for _ in range(20))
    suf = bytes(rng.choice(b"ACGT") for _ in range(20))
    seqs = make_reads(rng, pre, suf, 3000)
    for thr in (0.7, 0.8, 0.55, 0.95):
        table, diag, _ = gpu_run(seqs, (pre, suf), accept_prefix_alignment=thr, accept_suffix_alignment=thr)
        otable, odiag, _ = oracle_run(seqs, (pre, suf), accept_prefix_alignment=thr, accept_suffix_alignment=thr)
        assert_diag_equal(diag, odiag)
        assert table == otable
    assert any(s == 42 for s in odiag["score_prefix"]) or True


def test_skip_translation_and_invalid_utf8():
    rng = random.Random(10)
    seqs = make_reads(rng, PREFIX, SUFFIX, 500)
    pool = [b"\xff", b"\xc3\xa9", b"\xe2\x82\xac", b"\xf0\x9f\x98\x80", b"\xc0\x80", b"\xed\xa0\x80", b"\x80", b"A", b"CG"]
    for _ in range(300):
        mid = b"".join(rng.choice(pool) for _ in range(rng.randrange(1, 9)))
        seqs.append(PREFIX + mid + SUFFIX)
    for skip in (True, False):
        table, diag, _ = gpu_run(seqs, (PREFIX, SUFFIX), skip_translation=skip)
        otable, odiag, _ = oracle_run(seqs, (PREFIX, SUFFIX), skip_translation=skip)
        assert_diag_equal(diag, odiag)
        assert table == otable


def test_empty_and_degenerate_inputs():
    ad = (PREFIX, SUFFIX)
    assert gpu_run([], ad, want_diag=False)[0] == {}
    seqs = [b"", b"A", PREFIX, SUFFIX, PREFIX + SUFFIX, SUFFIX + PREFIX, PREFIX + b"A" + SUFFIX,
            PREFIX + b"ATG" + SUFFIX, b"", PREFIX + b"ATG" + SUFFIX + PREFIX + b"CCC" + SUFFIX,
            SUFFIX + b"AAA" + PREFIX + b"ATG" + SUFFIX]
    table, diag, _ = gpu_run(seqs, ad)
    otable, odiag, _ = oracle_run(seqs, ad)
    assert_diag_equal(diag, odiag)
    assert table == otable
    # batches of 64 reads: reads 320-447 and 832-895 make batches of empty reads only (no text at all), between
    # ordinary ones
    rng = random.Random(19)
    seqs = make_reads(rng, PREFIX, SUFFIX, 300) + [b""] * 200 + make_reads(rng, PREFIX, SUFFIX, 300) + [b""] * 100
    for skip in (False, True):
        table = gpu_run(seqs, ad, want_diag=False, batch_reads=64, skip_translation=skip)[0]
        assert table == oracle_run(seqs, ad, skip_translation=skip)[0]


def test_ragged_lengths_and_long_reads():
    rng = random.Random(11)
    seqs = []
    for _ in range(400):
        L = rng.choice([1, 5, 17, 18, 19, 40, 63, 64, 65, 127, 128, 129, 300, 700, 1500])
        body = bytearray(rng.choice(b"ACGT") for _ in range(L))
        if L > 60 and rng.random() < 0.8:
            a = mutate(rng, PREFIX)
            b = mutate(rng, SUFFIX)
            v = bytes(rng.choice(b"ACGT") for _ in range(21))
            ins = a + v + b
            p = rng.randrange(0, L - len(ins) + 1) if L > len(ins) else 0
            body[p:p + len(ins)] = ins
        seqs.append(bytes(body))
    table, diag, _ = gpu_run(seqs, (PREFIX, SUFFIX), accept_prefix_alignment=0.6, accept_suffix_alignment=0.6)
    otable, odiag, _ = oracle_run(seqs, (PREFIX, SUFFIX), accept_prefix_alignment=0.6, accept_suffix_alignment=0.6)
    assert_diag_equal(diag, odiag)
    assert table == otable


def test_gap_extend_zero_long_runs():
    # extend = 0: an extension run can be as long as the read (the x field of the packed word)
    rng = random.Random(12)
    seqs = [bytes(rng.choice(b"AC") for _ in range(rng.randrange(50, 400))) for _ in range(300)]
    seqs += make_reads(rng, PREFIX, SUFFIX, 300, lead=(0, 200))
    # longer than the packed word can count with extend == 0: goes through the fallback list
    seqs += [bytes(rng.choice(b"ACGT") for _ in range(L)) for L in (4090, 4100, 5000, 9000)]
    for sc in ((1, -1, 0, 0), (2, -1, 3, 0), (1, -3, 2, 0)):
        kw = dict(match_score=sc[0], mismatch_score=sc[1], gap_open_penalty=sc[2], gap_extend_penalty=sc[3])
        table, diag, _ = gpu_run(seqs, (PREFIX, SUFFIX), **kw)
        otable, odiag, _ = oracle_run(seqs, (PREFIX, SUFFIX), **kw)
        assert_diag_equal(diag, odiag)
        assert table == otable


def test_multi_batch_equals_single_batch():
    rng = random.Random(13)
    seqs = make_reads(rng, PREFIX, SUFFIX, 5000, lib=300)
    one = gpu_run(seqs, (PREFIX, SUFFIX), want_diag=False)[0]
    many = gpu_run(seqs, (PREFIX, SUFFIX), want_diag=False, batch_reads=257)[0]
    assert one == many == oracle_run(seqs, (PREFIX, SUFFIX))[0]


def test_suffix_dp_skip_does_not_change_the_table():
    rng = random.Random(14)
    seqs = make_reads(rng, PREFIX, SUFFIX, 4000)
    a, _, sa = gpu_run(seqs, (PREFIX, SUFFIX), want_diag=False)
    b, _, sb = gpu_run(seqs, (PREFIX, SUFFIX), want_diag=False, dp_compute_all=True)
    assert a == b == oracle_run(seqs, (PREFIX, SUFFIX))[0]
    assert sa["dp_suffix"] <= sb["dp_suffix"]


def test_hash_collisions_are_resolved_by_full_keys():
    rng = random.Random(15)
    seqs = make_reads(rng, PREFIX, SUFFIX, 6000, lib=2000)
    want = oracle_run(seqs, (PREFIX, SUFFIX))[0]
    for bits in (1, 4, 33):
        got = gpu_run(seqs, (PREFIX, SUFFIX), want_diag=False, debug_hash_bits=bits, batch_reads=1500)[0]
        assert got == want


def test_table_growth_many_uniques():
    rng = random.Random(16)
    n = 120000
    body = np.frombuffer(bytes(rng.choice(b"ACGT") for _ in range(n * 30)), dtype=np.uint8).reshape(n, 30)
    pre = np.frombuffer(PREFIX, dtype=np.uint8)
    suf = np.frombuffer(SUFFIX, dtype=np.uint8)
    reads = np.concatenate([np.tile(pre, (n, 1)), body, np.tile(suf, (n, 1))], axis=1)
    L = reads.shape[1]
    text = np.ascontiguousarray(reads).reshape(-1)
    off = np.arange(n, dtype=np.uint32) * L
    ln = np.full(n, L, dtype=np.uint32)
    with api.Context((PREFIX, SUFFIX), batch_reads=20000) as ctx:
        ctx.submit_host(text, spans_of(off, ln))
        got = ctx.finish_dict()
        st = ctx.stats()
    want, _, _ = oracle.process_reads(oracle.make_params((PREFIX, SUFFIX)), text, off, ln, n_threads=8)
    assert got == want
    assert st["unique"] == len(want) and st["counted"] == n


def test_partition_and_absorb_roundtrip():
    torch = pytest.importorskip("torch")
    rng = random.Random(17)
    seqs = make_reads(rng, PREFIX, SUFFIX, 8000, lib=900)
    text, off, ln = oracle.pack_reads(seqs)
    want = oracle_run(seqs, (PREFIX, SUFFIX))[0]
    with api.Context((PREFIX, SUFFIX)) as src:
        src.submit_host(text, spans_of(off, ln))
        for n_parts in (1, 3, 8):
            sizes = src.partition_sizes(n_parts)
            offs = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64)
            buf = torch.empty(int(sum(sizes)), dtype=torch.uint8, device="cuda")
            src.partition_fill(n_parts, buf.data_ptr(), offs)
            merged = {}
            for p in range(n_parts):
                with api.Context((PREFIX, SUFFIX)) as dst:
                    dst.absorb(buf.data_ptr() + int(offs[p]), sizes[p])
                    dst.absorb(buf.data_ptr() + int(offs[p]), sizes[p])      # counts add up
                    part = dst.finish_dict()
                assert not (set(part) & set(merged))                           # partitions are disjoint
                merged.update(part)
            assert merged == {k: 2 * v for k, v in want.items()}


def test_synth_device_matches_host_and_oracle():
    torch = pytest.importorskip("torch")
    cfg = api.synth_cfg(seed=1003, read_len=250, adapter_len=20, region_len=198, n_variants=5000,
                        p_err=0.30, indel=0.5, force_indel=1)
    n = 60000
    th, sh = api.synth_host(cfg, 1000, n)
    td = torch.empty(n * 250, dtype=torch.uint8, device="cuda")
    sd = torch.empty(n * 2, dtype=torch.int32, device="cuda")
    api.synth_device(cfg, 1000, n, td.data_ptr(), sd.data_ptr())
    assert (td.cpu().numpy() == th).all()
    assert (sd.cpu().numpy().view(np.uint32).reshape(n, 2) == np.stack([sh["off"], sh["len"]], 1)).all()
    ad = api.synth_adapters(cfg)
    with api.Context(ad, diagnostics=True, dp_compute_all=True) as ctx:
        ctx.submit_device(td.data_ptr(), td.numel(), sd.data_ptr(), n)
        diag = ctx.diag(n)
        got = ctx.finish_dict()
        st = ctx.stats()
    want, odiag, cells = oracle.process_reads(oracle.make_params(ad), th, sh["off"], sh["len"],
                                              n_threads=8, want_diag=True)
    assert_diag_equal(diag, odiag)
    assert got == want and st["dp_cells"] == cells
    assert st["dp_prefix"] > 0.2 * n and st["counted"] > 0.5 * n


def test_file_ingest_variants(tmp_path, golden):
    from conftest import write_fastq_gz
    from vfind_b200 import PanicException, find_variants
    toy = golden["toy"]
    reads = [(r["header"], r["seq"], r["qual"]) for r in toy["reads"]]
    ad = tuple(toy["adapters"])

    def rows(out):
        cols = out.to_pydict() if hasattr(out, "to_pydict") else out.to_dict(as_series=False)
        return dict(zip(cols["sequence"], cols["count"]))

    for kw in (dict(members=3), dict(crlf=True), dict(final_newline=False)):
        p = write_fastq_gz(tmp_path / "v.fq.gz", reads, **kw)
        assert rows(find_variants(str(p), ad)) == {"MAGICAL": 4}
    rng = random.Random(18)
    seqs = make_reads(rng, PREFIX, SUFFIX, 30000, lib=500)
    recs = [("r%d" % i, s.decode(), "F" * len(s)) for i, s in enumerate(seqs)]
    p = write_fastq_gz(tmp_path / "big.fq.gz", recs, members=5)
    got = rows(find_variants(str(p), (PREFIX.decode(), SUFFIX.decode()), accept_prefix_alignment=0.6))
    want = oracle.find_variants_file(str(p), (PREFIX, SUFFIX), n_threads=8, accept_prefix_alignment=0.6)
    assert {k.encode(): v for k, v in got.items()} == want
    # chunked ingest: records straddling chunk boundaries are carried over (tiny chunks force it)
    import os
    for chunk in ("700", "4096", "100000"):
        os.environ["VFB_INGEST_CHUNK"] = chunk
        try:
            got2 = rows(find_variants(str(p), (PREFIX.decode(), SUFFIX.decode()), accept_prefix_alignment=0.6))
        finally:
            del os.environ["VFB_INGEST_CHUNK"]
        assert got2 == got, chunk
    # a malformed record in the middle of a large file is reported with its index
    recs2 = list(recs)
    recs2[20000] = ("bad", "ACGT", "FFF")
    pb = write_fastq_gz(tmp_path / "bigbad.fq.gz", recs2, members=2)
    with pytest.raises(PanicException, match="record 20000"):
        find_variants(str(pb), ad)
    blank = tmp_path / "blank.fq.gz"
    import gzip as _gz
    blank.write_bytes(_gz.compress(b"@r\nACGT\n+\nFFFF\n\n\n\r\n"))
    assert rows(find_variants(str(blank), ad)) == {}
    mid = tmp_path / "mid.fq.gz"
    mid.write_bytes(_gz.compress(b"@r\nACGT\n+\nFFFF\n\n@q\nACGT\n+\nFFFF\n"))
    with pytest.raises(PanicException):
        find_variants(str(mid), ad)
    # empty file -> empty table with both columns (Q12)
    e = tmp_path / "e.fq.gz"
    import gzip
    e.write_bytes(gzip.compress(b""))
    out = find_variants(str(e), ad)
    assert rows(out) == {}
    # malformed inputs (the reference panics, src/lib.rs:308)
    bad = tmp_path / "bad.fq.gz"
    bad.write_bytes(gzip.compress(b"@r\nACGT\n+\nFFF\n"))
    with pytest.raises(PanicException):
        find_variants(str(bad), ad)
    plain = tmp_path / "plain.fq"
    plain.write_text("@r\nACGT\n+\nFFFF\n")
    with pytest.raises(PanicException):
        find_variants(str(plain), ad)
    trunc = tmp_path / "trunc.fq.gz"
    trunc.write_bytes(gzip.compress(b"@r\nACGT\n+\nFFFF\n@q\nAC"))
    with pytest.raises(PanicException):
        find_variants(str(trunc), ad)


def test_arrow_c_data_export_is_zero_copy_and_outlives_the_context():
    # SURVEY §8(f) next-2: the result table leaves through the Arrow C Data Interface
    import gc
    import pyarrow as pa
    rng = random.Random(21)
    seqs = make_reads(rng, PREFIX, SUFFIX, 6000, lib=700)
    text, off, ln = oracle.pack_reads(seqs)
    want = oracle_run(seqs, (PREFIX, SUFFIX))[0]
    with api.Context((PREFIX, SUFFIX)) as ctx:
        ctx.submit_host(text, spans_of(off, ln))
        batch = ctx.finish_arrow()
        # the context stays usable and hands out fresh columns next time
        ctx.submit_host(text, spans_of(off, ln))
        twice = ctx.finish_dict()
    assert batch.schema.names == ["sequence", "count"]
    assert batch.schema.field("sequence").type == pa.large_string() and batch.schema.field("count").type == pa.uint64()
    assert batch.num_rows == len(want)
    got = {k.encode(): v for k, v in zip(batch.column(0).to_pylist(), batch.column(1).to_pylist())}
    assert got == want                                   # read after the context is gone
    assert twice == {k: 2 * v for k, v in want.items()}
    frame = api.batch_to_frame(batch)
    cols = frame.to_pydict() if hasattr(frame, "to_pydict") else frame.to_dict(as_series=False)
    assert {k.encode(): v for k, v in zip(cols["sequence"], cols["count"])} == want
    # zero-copy: the Arrow buffers are not owned by Python (they are the pinned columns)
    data_buf = batch.column(0).buffers()[2]
    assert data_buf.size >= sum(len(k) for k in want) and data_buf.address != 0
    del batch, frame, cols, data_buf
    gc.collect()                                         # release callback -> pinned pool, no crash
    # empty result (Q12): both columns, zero rows
    with api.Context((PREFIX, SUFFIX)) as ctx:
        empty = ctx.finish_arrow()
    assert empty.num_rows == 0 and empty.schema.names == ["sequence", "count"]


@pytest.mark.parametrize("skip", [False, True])
def test_fused_key_count_kernel_matches_separate_kernels(monkeypatch, skip):
    """k34_keys_count (the key kernel probes the table and counts reads whose key already has a row; only the rest
    go through k4_insert / k4_publish) against K3 + K4 over every read (VFB_FUSED_COUNT=0) and the oracle:
    many small batches, so that later batches find most of their keys in the table; regions with lower case, U, N,
    '-' and non-ASCII bytes (the arithmetic translate must hand those groups to the per-byte tables)."""
    rng = random.Random(41)
    seqs = make_reads(rng, PREFIX, SUFFIX, 24000, lib=700, alphabet=b"ACGTACGTACGTACGTacgtUuN-")
    seqs += make_reads(rng, PREFIX, SUFFIX, 2000, lib=50, alphabet=b"ACGT\xc3\xa9\xff")
    rng.shuffle(seqs)
    kw = dict(want_diag=False, skip_translation=skip, batch_reads=1500)
    want = oracle_run(seqs, (PREFIX, SUFFIX), skip_translation=skip)[0]
    fused, _, sf = gpu_run(seqs, (PREFIX, SUFFIX), **kw)
    assert fused == want
    # (the first batch meets an empty table and goes through the separate kernels)
    assert sf["fused_batches"] == (len(seqs) + 1499) // 1500 - 1 and 0 < sf["fused_hits"] < sf["counted"]
    assert sf["counted"] == sum(want.values()) and sf["unique"] == len(want)
    monkeypatch.setenv("VFB_FUSED_COUNT", "0")
    plain, _, sp = gpu_run(seqs, (PREFIX, SUFFIX), **kw)
    assert plain == want and sp["fused_batches"] == 0 and sp["fused_hits"] == 0
    monkeypatch.delenv("VFB_FUSED_COUNT")
    # forced hash collisions: long probe chains leave the fused kernel and are settled by the insert kernels
    for bits in (1, 5):
        got, _, st = gpu_run(seqs, (PREFIX, SUFFIX), debug_hash_bits=bits, **kw)
        assert got == want and st["counted"] == sum(want.values())


def test_fused_key_count_second_pass_is_all_hits():
    """The same reads twice through one context: every key of the second pass already has a row, so the fused
    kernel counts all of them itself and the counts double."""
    rng = random.Random(42)
    seqs = make_reads(rng, PREFIX, SUFFIX, 9000, lib=400)
    text, off, ln = oracle.pack_reads(seqs)
    want = oracle_run(seqs, (PREFIX, SUFFIX))[0]
    with api.Context((PREFIX, SUFFIX), batch_reads=3000) as ctx:
        ctx.submit_host(text, spans_of(off, ln))
        ctx.sync()
        first = ctx.stats()
        ctx.submit_host(text, spans_of(off, ln))
        got = ctx.finish_dict()
        st = ctx.stats()
    assert got == {k: 2 * v for k, v in want.items()}
    assert st["unique"] == first["unique"] == len(want)
    assert st["fused_hits"] - first["fused_hits"] == sum(want.values())
