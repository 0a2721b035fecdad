"""collapse_ratio without a GPU: the reference against its brute-force form, the properties of the result, argument
validation on every entry point, and the ABI structs."""
import ctypes
import inspect
import math
import random

import numpy as np
import pytest

import collapse_oracle as co
from vfind_b200 import api

ALPHABETS = [b"ACGT", b"ACGTN", b"ACDEFGHIKLMNPQRSTVWY*X", bytes([0x00, 0xFF, 0x41])]
RATIOS = [1, 1.5, 2, 10, 1e300]


def mutate(rng, key, alphabet):
    p = rng.randrange(len(key))
    x = rng.choice([b for b in alphabet if b != key[p]])
    return key[:p] + bytes([x]) + key[p + 1:]


def random_table(rng, alphabet, n_parents=None):
    """Parents with error tails: single-substitution stars, chains of substitutions, tied counts, a few zero counts and
    keys of other lengths."""
    table = {}
    L = rng.choice((1, 2, 3, 5, 8))
    n_parents = n_parents or rng.randrange(1, 6)
    for _ in range(n_parents):
        k = bytes(rng.choice(alphabet) for _ in range(L + rng.choice((0, 0, 0, 1))))
        table[k] = rng.choice((1, 2, 5, 10, 100, 1000))
        cur = k
        for _ in range(rng.randrange(0, 8)):
            shape = rng.randrange(3)
            base = cur if shape == 0 else k                  # 0: a chain, else a star around the parent
            m = mutate(rng, base, alphabet)
            if m not in table:
                table[m] = rng.choice((1, 1, 2, 3, 5, table.get(base, 1), max(1, table.get(base, 1) // 2)))
            cur = m
    for k in list(table)[:rng.randrange(0, 2)]:
        if rng.random() < 0.3:
            table[k] = 0
    return table


@pytest.mark.parametrize("alphabet", ALPHABETS, ids=["dna", "dna_n", "protein", "bytes"])
def test_reference_matches_brute_force(alphabet):
    rng = random.Random(hash(alphabet) & 0xFFFF)
    for _ in range(800):
        t = random_table(rng, alphabet)
        r = rng.choice(RATIOS)
        want = co.collapse_brute_force(t, r)
        got = co.collapse_reference(t, r)
        assert got == want, (t, r)
        assert sum(got.values()) == sum(t.values())
        assert set(got) == co.roots(t, r)
        assert all(v > 0 for v in got.values())


def test_hand_built_cases():
    # a chain: AAAA <- AAAC <- AACC (two substitutions from its root, folded through the middle row)
    assert co.collapse_reference({b"AAAA": 100, b"AAAC": 10, b"AACC": 2}, 2) == {b"AAAA": 112}
    # the middle row fails the ratio against the root: two clusters
    assert co.collapse_reference({b"AAAA": 100, b"AAAC": 60, b"AACC": 2}, 2) == {b"AAAA": 100, b"AAAC": 62}
    # tie on count: the smaller key comes first and is the parent at ratio 1, never at ratio > 1
    assert co.collapse_reference({b"AC": 5, b"AG": 5}, 1) == {b"AC": 10}
    assert co.collapse_reference({b"AC": 5, b"AG": 5}, 1.5) == {b"AC": 5, b"AG": 5}
    # exactly at ratio * count qualifies
    assert co.collapse_reference({b"AC": 10, b"AG": 5}, 2) == {b"AC": 15}
    assert co.collapse_reference({b"AC": 9, b"AG": 5}, 2) == {b"AC": 9, b"AG": 5}
    # two candidate parents: the first in the order wins (count, then key bytes, unsigned)
    t = {b"\xffB": 50, b"\x00B": 50, b"AB": 1}
    assert co.collapse_reference(t, 2) == {b"\x00B": 51, b"\xffB": 50}
    # different lengths are never neighbours; count 0 rows vanish
    assert co.collapse_reference({b"A": 9, b"AA": 1, b"C": 0}, 1) == {b"A": 9, b"AA": 1}
    # a ratio no pair reaches leaves the table as it is
    t = {b"AAAA": 2 ** 60, b"AAAC": 1}
    assert co.collapse_reference(t, 1e300) == t
    assert co.collapse_reference({}, 2) == {}


def test_float_semantics_of_the_ratio():
    # counts past 2^53: float() rounds to nearest, as the library's u64 -> double conversion does
    a, b = 2 ** 53 + 1, 2 ** 52
    assert float(a) >= 2.0 * float(b)              # 2^53 + 1 rounds down to 2^53
    assert co.collapse_reference({b"AA": a, b"AC": b}, 2) == {b"AA": a + b}
    assert co.collapse_reference({b"AA": 2 ** 53 - 1, b"AC": 2 ** 52}, 2) == {b"AA": 2 ** 53 - 1, b"AC": 2 ** 52}


def test_result_does_not_depend_on_row_order():
    rng = random.Random(5)
    for _ in range(200):
        t = random_table(rng, b"ACGT")
        items = list(t.items())
        rng.shuffle(items)
        assert co.collapse_reference(dict(items), 2) == co.collapse_reference(t, 2)


BAD_RATIOS = [0.5, 0.0, -1, float("nan"), float("inf"), -float("inf")]


def test_collapse_ratio_validation_on_every_entry_point(tmp_path):
    f = tmp_path / "missing.fq.gz"             # validation comes before the file is opened
    ad = ("ACGT", "TTGA")
    for fn in (lambda r: api.find_variants(str(f), ad, collapse_ratio=r),
               lambda r: api.find_variants_multi([str(f)], ad, collapse_ratio=r),
               lambda r: api.Context(ad, collapse_ratio=r),
               lambda r: api.MultiContext(ad, collapse_ratio=r),
               lambda r: api.collapse_variants({"sequence": [], "count": []}, r)):
        for r in BAD_RATIOS:
            with pytest.raises(ValueError):
                fn(r)
        for r in (True, False, "2", [2], 2j):
            with pytest.raises(TypeError):
                fn(r)
    with pytest.raises(TypeError):
        api.collapse_variants({"sequence": [], "count": []}, None)
    for f_ in (api.find_variants, api.find_variants_multi, api.Context, api.MultiContext):
        prm = inspect.signature(f_).parameters["collapse_ratio"]
        assert prm.kind is inspect.Parameter.KEYWORD_ONLY and prm.default is None
    assert inspect.signature(api.collapse_variants).parameters["device"].kind is inspect.Parameter.KEYWORD_ONLY
    assert api._ratio_arg(None, "r", True) == 0.0 and api._ratio_arg(np.int64(3), "r", False) == 3.0


def test_collapse_variants_rejects_other_inputs():
    import pyarrow as pa
    with pytest.raises(TypeError):
        api.collapse_variants({"sequence": [b"A"], "count": [1]}, 2)
    with pytest.raises(TypeError):
        api.collapse_variants(pa.table({"sequence": [1], "count": [1]}), 2)
    with pytest.raises(ValueError):
        api.collapse_variants(pa.table({"sequence": ["A"], "count": [-1]}), 2)
    with pytest.raises(ValueError):
        api.collapse_variants(pa.table({"sequence": ["A", None], "count": [1, 2]}), 2)


def test_library_validates_the_ratio_before_any_device_use():
    lib = api.load_library()
    ad = (b"ACGT", b"TTGA")
    for r in (0.5, float("nan"), float("inf"), -1.0):
        p, _, _ = api._make_params(lib, ad, 3, -2, 5, 2, 0.75, 0.75, 3, 2, False, False, None, False, 0, 0, 0, 0,
                                   False, False, False, 0, 0)
        p.collapse_ratio = r
        h = ctypes.c_void_p()
        assert lib.vfb_create(ctypes.byref(p), ctypes.byref(h)) == api.VFB_ERR_VALUE
        t_in, t_out = api.Table(), api.Table()
        assert lib.vfb_collapse(ctypes.byref(t_in), r, -1, 0, ctypes.byref(t_out), None) == api.VFB_ERR_VALUE
    assert lib.vfb_collapse(None, 2.0, -1, 0, None, None) == api.VFB_ERR_ARG


def test_new_structs_match_the_header():
    lib = api.load_library()
    p = api.Params()
    lib.vfb_default_params(ctypes.byref(p))
    assert p.struct_size == ctypes.sizeof(api.Params) and p.collapse_ratio == 0.0
    assert [f for f, _ in api.Params._fields_][-1] == "collapse_ratio"
    assert api.Params.collapse_ratio.offset == ctypes.sizeof(api.Params) - 8
    assert ctypes.sizeof(api.CollapseInfo) == 24 and [f for f, _ in api.CollapseInfo._fields_] == ["rows_in", "rows_out", "ms"]
    for name in ("vfb_collapse", "vfb_get_collapse_info", "vfb_multi_get_collapse_info"):
        assert hasattr(lib, name)
    assert [f for f, _ in api.Stats._fields_][-1] == "reverse_counted"      # vfb_stats did not grow
    import vfind
    assert "collapse_variants" in api.__dict__ and "collapse_variants" not in vfind.__all__
    assert not math.isnan(p.collapse_ratio)
