"""both_strands without a GPU: the reverse complement, the oracle's two-pass composition and the ABI structs."""
import ctypes

import numpy as np
import pytest

import oracle
import strand_oracle
from vfind_b200 import api

PREFIX = b"GGGCCCAGCCGGCCGGAT"
SUFFIX = b"CCGGAGGCGGAGGTTCAG"
REGION = b"ATGGCTAGCAAAGGAGAAGAA"          # 21 bases: MASKGEE


def test_reverse_complement_map():
    for rc in (strand_oracle.revcomp, api.reverse_complement):
        assert rc(b"ACGTacgt") == b"acgtACGT"
        assert rc(rc(b"ACGTTGCAacgtgcaAT")) == b"ACGTTGCAacgtgcaAT"
        assert rc(b"U") == b"A" and rc(b"u") == b"a" and rc(b"UuAa") == b"tTaA"
        other = bytes(b for b in range(256) if b not in b"ACGTUacgtu")
        assert rc(other) == other[::-1]
        assert rc(b"") == b""


def test_library_reverse_complement_matches_the_oracle():
    lib = api.load_library()
    every = bytes(range(256)) + b"ACGTUacgtuNn-"
    out = ctypes.create_string_buffer(len(every))
    assert lib.vfb_debug_revcomp(every, len(every), out) == 0
    assert out.raw == strand_oracle.revcomp(every)


def _both(seqs, **kw):
    text, off, ln = oracle.pack_reads(seqs)
    return strand_oracle.process_reads_both_strands(oracle.make_params((PREFIX, SUFFIX), **kw), text, off, ln, want_diag=True)


def test_toy_reads_reverse_complemented(golden):
    toy = golden["toy"]
    ad = tuple(a.encode() for a in toy["adapters"])
    seqs = [strand_oracle.revcomp(r["seq"].encode()) for r in toy["reads"]]
    text, off, ln = oracle.pack_reads(seqs)
    p = oracle.make_params(ad)
    assert oracle.process_reads(p, text, off, ln)[0] == {}
    table, fdiag, rdiag, cells = strand_oracle.process_reads_both_strands(p, text, off, ln, want_diag=True)
    assert table == {b"MAGICAL": 4}
    assert cells >= oracle.process_reads(p, text, off, ln)[2]


def test_read_with_regions_on_both_strands_counts_once_forward():
    other = b"ATGCCCGGGAAATTTCCCGGG"          # MPGKFPG
    read = PREFIX + REGION + SUFFIX + strand_oracle.revcomp(PREFIX + other + SUFFIX)
    table, fdiag, rdiag, _ = _both([read])
    assert table == {oracle.translate(REGION): 1}
    assert rdiag["start"][0] == -1 and rdiag["score_prefix"][0] == oracle.INT32_MIN   # not retried
    # the reverse pass alone would have found the other region
    table_rc, _, _, _ = _both([strand_oracle.revcomp(PREFIX + other + SUFFIX)])
    assert table_rc == {oracle.translate(other): 1}


def test_forward_region_of_partial_codons_is_not_retried():
    read = PREFIX + REGION + b"A" + SUFFIX + strand_oracle.revcomp(PREFIX + REGION + SUFFIX)
    table, fdiag, rdiag, _ = _both([read])
    assert strand_oracle.has_region(fdiag, [len(read)])[0]
    assert table == {}
    assert rdiag["exact_prefix"][0] == -1 and rdiag["start"][0] == -1
    # with skip_translation the same forward region is counted as it stands
    table, _, _, _ = _both([read], skip_translation=True)
    assert table == {REGION + b"A": 1}


def test_suffix_length_past_the_read_is_retried():
    # a read made of the suffix adapter with one base deleted: the alignment is accepted, its length statistic (18)
    # exceeds the read (17 bases), so no boundary comes of it (Q8) and the read has no forward region
    read = SUFFIX[:9] + SUFFIX[10:]
    table, fdiag, rdiag, _ = _both([read])
    assert fdiag["score_suffix"][0] > 0.75 * 3 * len(SUFFIX) and fdiag["len_suffix"][0] > len(read)
    assert fdiag["end"][0] == -1 and not strand_oracle.has_region(fdiag, [len(read)])[0]
    assert rdiag["score_prefix"][0] != oracle.INT32_MIN            # the reverse pass ran
    assert table == {}


def test_empty_reads_are_not_retried_and_reverse_rows_keep_read_order():
    fwd = PREFIX + REGION + SUFFIX
    seqs = [b"", strand_oracle.revcomp(fwd), fwd, b"", b"NNNN", strand_oracle.revcomp(fwd)]
    table, fdiag, rdiag, _ = _both(seqs)
    assert table == {oracle.translate(REGION): 3}
    ran = rdiag["exact_prefix"] >= 0
    assert list(ran) == [False, True, False, False, False, True]
    assert rdiag["start"][4] == -1 and rdiag["score_prefix"][4] != oracle.INT32_MIN   # retried, nothing found
    assert rdiag["score_prefix"][0] == oracle.INT32_MIN and rdiag["len_prefix"][3] == -1


def test_new_structs_match_the_header():
    lib = api.load_library()
    p = api.Params()
    lib.vfb_default_params(ctypes.byref(p))
    assert p.struct_size == ctypes.sizeof(api.Params) and p.both_strands == 0
    fields = [f for f, _ in api.Stats._fields_]
    assert fields[-2:] == ["reverse_reads", "reverse_counted"]
    assert ctypes.sizeof(api.Stats) == api.Stats.reverse_counted.offset + 8
    assert api.DIAG_DTYPE.itemsize == 32
    assert hasattr(lib, "vfb_get_diag_reverse")


def test_keyword_only_argument():
    import inspect

    import vfind
    for f in (api.find_variants, api.find_variants_multi, api.Context, api.MultiContext, api.read_diagnostics):
        prm = inspect.signature(f).parameters["both_strands"]
        assert prm.kind is inspect.Parameter.KEYWORD_ONLY and prm.default is False
    with pytest.raises(TypeError):
        api.find_variants("x.fq.gz", ("A", "C"), 3, -2, 5, 2, 0.75, 0.75, 3, 2, False, True, False)
    assert "both_strands" not in list(inspect.signature(vfind.find_variants).parameters)[:12]
    assert np.dtype(api.SPAN_DTYPE).itemsize == 8
