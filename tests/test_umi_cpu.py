"""umi_length without a GPU: the reference on hand-built reads, argument validation and the ABI."""
import ctypes

import pytest

import oracle
import strand_oracle
import umi_oracle
from vfind_b200 import api

PREFIX = b"GGGCCCAGCCGGCCGGAT"
SUFFIX = b"CCGGAGGCGGAGGTTCAG"
V1 = b"ATGGCTAGCAAAGGAGAAGAA"          # MASKGEE
V2 = b"ATGGCTAGCAAAGGAGAAGAG"          # MASKGEE as well (GAG = E): same key as V1 when translating
V3 = b"ATGTTTAGCAAAGGAGAAGAA"          # MFSKGEE


def read(umi, region, tail=b"TT"):
    return umi + PREFIX + region + SUFFIX + tail


def params(**kw):
    return oracle.make_params((PREFIX, SUFFIX), **kw)


def test_one_molecule_read_many_times():
    got, short, pairs = umi_oracle.umi_reads([read(b"ACGTACGTAC", V1)] * 7, params(), 10)
    assert got == {b"MASKGEE": (7, 1)} and short == 0 and pairs == 1


def test_one_umi_under_two_variants():
    seqs = [read(b"AAAACCCCGG", V1)] * 3 + [read(b"AAAACCCCGG", V3)] * 2
    got, short, pairs = umi_oracle.umi_reads(seqs, params(), 10)
    assert got == {b"MASKGEE": (3, 1), b"MFSKGEE": (2, 1)} and pairs == 2


def test_one_variant_under_many_umis():
    umis = [bytes(b"ACGT"[(i >> (2 * j)) & 3] for j in range(6)) for i in range(50)]
    seqs = [read(u, V1) for u in umis] + [read(umis[0], V2)]       # V2 translates to the same key
    got, _, pairs = umi_oracle.umi_reads(seqs, params(), 6)
    assert got == {b"MASKGEE": (51, 50)} and pairs == 50
    got, _, _ = umi_oracle.umi_reads(seqs, params(skip_translation=True), 6)
    assert got == {V1: (50, 50), V2: (1, 1)}


def test_reads_one_byte_too_short():
    r = read(b"", V1, tail=b"")                                   # UMI taken from the end of the read
    n = len(r)
    got, short, _ = umi_oracle.umi_reads([r, r + b"G"], params(), 4, umi_offset=n - 3)
    assert short == 1 and got == {b"MASKGEE": (1, 1)}
    got, short, _ = umi_oracle.umi_reads([r, r + b"G"], params(), 3, umi_offset=n - 3)
    assert short == 0 and got == {b"MASKGEE": (2, 1)}               # both end in the same three bytes
    # a read without a key is neither counted nor short
    got, short, _ = umi_oracle.umi_reads([b"AC" + PREFIX + V1[:-1] + SUFFIX], params(), 50)
    assert got == {} and short == 0


def test_umis_with_n_and_lower_case_are_raw_bytes():
    seqs = [read(b"ACGNN", V1), read(b"acgnn", V1), read(b"ACGNN", V1), read(b"ACGnN", V1)]
    got, _, pairs = umi_oracle.umi_reads(seqs, params(), 5)
    assert got == {b"MASKGEE": (4, 3)} and pairs == 3


def test_reverse_counted_read_takes_its_umi_from_the_reverse_complement():
    fwd = read(b"AAAAACCCCC", V1)
    rev = strand_oracle.revcomp(read(b"GGGGGTTTTT", V1))
    got, _, _ = umi_oracle.umi_reads([fwd, rev], params(), 10, both_strands=True)
    assert got == {b"MASKGEE": (2, 2)}
    # the same physical UMI in both orientations is one molecule
    got, _, _ = umi_oracle.umi_reads([fwd, strand_oracle.revcomp(fwd)], params(), 10, both_strands=True)
    assert got == {b"MASKGEE": (2, 1)}
    # without both_strands the reverse read has no region
    got, _, _ = umi_oracle.umi_reads([fwd, rev], params(), 10)
    assert got == {b"MASKGEE": (1, 1)}


def test_umi_argument_validation_on_every_entry_point(tmp_path):
    ad = ("ACGT", "TTGA")
    missing = str(tmp_path / "missing.fq.gz")
    for fn in (lambda **kw: api.find_variants(missing, ad, **kw),
               lambda **kw: api.find_variants_multi([missing], ad, **kw)):
        for bad in ("10", 1.5, [3]):
            with pytest.raises(TypeError):
                fn(umi_length=bad)
            with pytest.raises(TypeError):
                fn(umi_length=8, umi_offset=bad)
        for length, offset in ((0, 0), (65, 0), (-1, 0), (8, -1), (8, 65529), (None, 3)):
            with pytest.raises(ValueError):
                fn(umi_length=length, umi_offset=offset)
        # rejected before the (missing) file is opened
        with pytest.raises(ValueError):
            fn(umi_length=8, collapse_ratio=2.0)
        with pytest.raises(FileNotFoundError):
            fn(umi_length=64, umi_offset=65472)
    for cls in (api.Context, api.MultiContext):
        with pytest.raises(ValueError):
            cls(ad, umi_length=8, collapse_ratio=2.0)
        with pytest.raises(ValueError):
            cls(ad, umi_length=65)
        with pytest.raises(TypeError):
            cls(ad, umi_length="8")
    with pytest.raises(ValueError):
        api.read_diagnostics([b"ACGT"], ad, umi_length=0)
    with pytest.raises(TypeError):
        api.read_diagnostics([b"ACGT"], ad, umi_length=2.0)


def test_library_validates_umi_values_before_any_device_use():
    lib = api.load_library()
    for off, length in ((0, 65), (65500, 64), (1, 0), (0xFFFFFFFF, 1)):
        assert lib.vfb_set_umi(None, off, length) == api.VFB_ERR_VALUE
        assert lib.vfb_multi_set_umi(None, off, length) == api.VFB_ERR_VALUE
    assert lib.vfb_set_umi(None, 0, 8) == api.VFB_ERR_ARG
    assert lib.vfb_multi_set_umi(None, 0, 8) == api.VFB_ERR_ARG
    info = api.UmiInfo()
    assert lib.vfb_get_umi_info(None, ctypes.byref(info)) == api.VFB_ERR_ARG
    col = ctypes.POINTER(ctypes.c_uint64)()
    assert lib.vfb_get_molecules(None, ctypes.byref(col)) == api.VFB_ERR_ARG


def test_new_structs_match_the_header():
    assert ctypes.sizeof(api.UmiInfo) == 32
    assert [f for f, _ in api.UmiInfo._fields_] == ["pairs", "rows_out", "reads_short", "ms"]
    lib = api.load_library()
    for name in ("vfb_set_umi", "vfb_get_umi_info", "vfb_get_molecules", "vfb_multi_set_umi", "vfb_multi_get_umi_info",
                 "vfb_multi_get_molecules"):
        assert hasattr(lib, name)
    assert [f for f, _ in api.Params._fields_][-1] == "collapse_ratio"       # vfb_params did not grow
    assert [f for f, _ in api.Stats._fields_][-1] == "reverse_counted"       # vfb_stats did not grow
