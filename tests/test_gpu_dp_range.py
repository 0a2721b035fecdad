"""GPU parity of the packed DP at scorings where the packed word has the least room (tests/test_packed_dp_model_cpu.py
models the word on the CPU; this runs the kernels).

A window of the windowed path starts from -inf in every row, so its cells reach lower scores than the full matrix's;
a layout sized for the full matrix only wrapped int32 there and accepted alignments with wrong scores and lengths.
Each point runs the windowed path per read with diagnostics (dp_mode=2), the default table and the full DP
(dp_mode=1) against the oracle, on reads with junk that mismatches the adapter on shifted diagonals in front of it,
and checks that the context picks the kernel vfb_debug_dp_layout predicts.  Reads of exactly the longest length the
packed layout takes, and one base longer, check the hand-over to the unpacked kernel.
"""
import random

import pytest

from test_gpu_parity import mutate
from test_gpu_windowed import check_windowed
from test_packed_dp_model_cpu import diagonal_junk, layout, lib  # noqa: F401  (lib: the module's fixture)

pytestmark = pytest.mark.gpu

POINTS = [((2, -2, 5, 5), 20, 0.75), ((3, -3, 6, 6), 16, 0.8), ((10, -9, 7, 7), 12, 0.75), ((4, -7, 10, 12), 32, 0.8),
          ((4, -7, 10, 12), 64, 0.8), ((1, -2, 3, 3), 12, 0.75), ((1, -2, 3, 3), 24, 0.75), ((3, -2, 4, 4), 8, 0.75),
          ((3, -2, 5, 2), 33, 0.8), ((2, -3, 4, 1), 20, 0.75), ((1, -1, 4, 4), 64, 0.9), ((5, -4, 10, 1), 33, 0.85),
          ((9, -10, 15, 15), 64, 0.9)]


def scoring_kw(sc, thr):
    return dict(match_score=sc[0], mismatch_score=sc[1], gap_open_penalty=sc[2], gap_extend_penalty=sc[3],
                accept_prefix_alignment=thr, accept_suffix_alignment=thr)


def expected_kind(lib, sc, thr, adapters):
    lays = [layout(lib, sc, len(a), thr) for a in adapters]
    if any(lay["packed"] and lay["max_edits"] >= 0 for lay in lays):
        return 3
    return 1 if any(lay["packed"] for lay in lays) else 2


def junk_reads(rng, pre, suf, n, K):
    """prefix ... region ... suffix, each adapter with up to K + 2 edits behind A + K bases of diagonal junk, some cut by
    a read end."""
    A = len(pre)
    seqs = []
    for it in range(n):
        a = mutate(rng, pre, max_edits=K + 2)
        b = mutate(rng, suf, max_edits=K + 2)
        region = bytes(rng.choice(b"ACGT") for _ in range(rng.choice((21, 24, 30))))
        read = diagonal_junk(rng, pre, A + K + rng.randrange(0, A)) + a + region + diagonal_junk(rng, suf, rng.randrange(0, A)) + b
        read += bytes(rng.choice(b"ACGT") for _ in range(rng.randrange(0, 12)))
        if it % 5 == 1:
            read = read[: len(read) - rng.randrange(1, max(2, A // 4))]
        elif it % 5 == 2:
            read = a[rng.randrange(1, max(2, A // 4)):] + region + b
        seqs.append(read)
    return seqs


@pytest.mark.parametrize("sc,A,thr", POINTS)
def test_packed_range_scorings(lib, sc, A, thr):
    rng = random.Random(hash((sc, A, thr)) & 0xFFFF)
    pre = bytes(rng.choice(b"ACGT") for _ in range(A))
    suf = bytes(rng.choice(b"ACGT") for _ in range(A))
    K = max(layout(lib, sc, A, thr)["max_edits"], 3)
    seqs = junk_reads(rng, pre, suf, 2500, K)
    kind = expected_kind(lib, sc, thr, (pre, suf))
    st = check_windowed(seqs, (pre, suf), expect_windowed=kind == 3, **scoring_kw(sc, thr))
    assert st["dp_kernel_kind"] == kind


@pytest.mark.parametrize("sc,A,thr", [((10, -10, 8, 8), 64, 0.9), ((10, -10, 15, 0), 64, 0.75)])
def test_reads_at_the_packed_length_cap(lib, sc, A, thr):
    """Large scores leave few bits for the length: reads of lcap bases run packed, reads of lcap + 1 go to the unpacked
    kernel (from the filter and from the full kernel), with the same results."""
    rng = random.Random(A + sc[2])
    pre = bytes(rng.choice(b"ACGT") for _ in range(A))
    suf = bytes(rng.choice(b"ACGT") for _ in range(A))
    caps = {layout(lib, sc, A, thr)["lcap"], layout(lib, sc, A, thr, dp_mode=1)["lcap"]}
    assert all(c < 4096 for c in caps), caps
    seqs = []
    for cap in sorted(caps):
        for L in (cap - 1, cap, cap + 1):
            for k in range(6):
                core = mutate(rng, pre, 3) + bytes(rng.choice(b"ACGT") for _ in range(24)) + mutate(rng, suf, 3)
                if k % 3 == 2:
                    core = core[: len(core) - 5]                    # suffix over the read's end
                lead = rng.randrange(0, L - len(core) + 1)
                body = diagonal_junk(rng, pre, lead) + core
                seqs.append((body + bytes(rng.choice(b"ACGT") for _ in range(L - len(body))))[:L])
    seqs += junk_reads(rng, pre, suf, 200, 6)
    kind = expected_kind(lib, sc, thr, (pre, suf))
    st = check_windowed(seqs, (pre, suf), expect_windowed=kind == 3, **scoring_kw(sc, thr))
    assert st["dp_kernel_kind"] == kind
