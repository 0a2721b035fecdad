"""both_strands on the GPU against the oracle's two-pass composition (tests/strand_oracle.py), bit for bit:
table, counted reads, DP cells, reverse_reads / reverse_counted, and the forward and reverse per-read diagnostics."""
import gzip
import random

import numpy as np
import pytest

import oracle
import strand_oracle
from vfind_b200 import api

pytestmark = pytest.mark.gpu

PREFIX = b"GGGCCCAGCCGGCCGGAT"
SUFFIX = b"CCGGAGGCGGAGGTTCAG"
ODD = bytes([0xC3, 0xA9, 0xE2, 0x82, 0xAC])          # multi-byte UTF-8 that reversal breaks up


def spans_of(off, ln):
    s = np.zeros(len(off), dtype=api.SPAN_DTYPE)
    s["off"], s["len"] = off, ln
    return s


def mutate(rng, ad, max_edits=3):
    inst = bytearray(ad)
    for _ in range(rng.randrange(0, max_edits + 1)):
        k = rng.randrange(len(inst))
        op = rng.randrange(3)
        if op == 0:
            inst[k] = rng.choice(b"ACGT")
        elif op == 1 and len(inst) > 1:
            del inst[k]
        else:
            inst.insert(k, rng.choice(b"ACGT"))
    return bytes(inst)


def make_reads(rng, pre, suf, n, alphabet=b"ACGT", lib=24, empty=0.0):
    """Forward reads, reverse-complemented reads, reads with a region on both strands and reads with none."""
    variants = [bytes(rng.choice(alphabet) for _ in range(rng.choice((21, 21, 24, 22, 30)))) for _ in range(lib)]
    junk = lambda k: bytes(rng.choice(alphabet) for _ in range(k))
    seqs = []
    for _ in range(n):
        u = rng.random()
        if u < empty:
            seqs.append(b"")
            continue
        one = lambda: (pre if rng.random() < 0.5 else mutate(rng, pre)) + rng.choice(variants) + \
            (suf if rng.random() < 0.5 else mutate(rng, suf))
        kind = rng.randrange(5)
        if kind == 0:
            r = one()
        elif kind in (1, 2):
            r = strand_oracle.revcomp(one())
        elif kind == 3:
            r = one() + junk(rng.randrange(0, 5)) + strand_oracle.revcomp(one())
        else:
            r = junk(rng.randrange(10, 90))
        seqs.append(junk(rng.randrange(0, 7)) + r + junk(rng.randrange(0, 7)))
    return seqs


def expected(seqs, adapters, **kw):
    okw = {k: v for k, v in kw.items() if k in ("match_score", "mismatch_score", "gap_open_penalty", "gap_extend_penalty",
                                                "accept_prefix_alignment", "accept_suffix_alignment", "skip_translation")}
    text, off, ln = oracle.pack_reads(seqs)
    p = oracle.make_params(adapters, **okw)
    table, fdiag, rdiag, cells = strand_oracle.process_reads_both_strands(p, text, off, ln, n_threads=8, want_diag=True)
    fwd_table = oracle.process_reads(p, text, off, ln, n_threads=8)[0]
    retried = ~strand_oracle.has_region(fdiag, ln) & (ln > 0)
    return dict(table=table, fdiag=fdiag, rdiag=rdiag, cells=cells, counted=sum(table.values()),
                reverse_reads=int(retried.sum()), reverse_counted=sum(table.values()) - sum(fwd_table.values()))


def gpu_run(seqs, adapters, diag=False, **kw):
    text, off, ln = oracle.pack_reads(seqs)
    with api.Context(adapters, diagnostics=diag, both_strands=True, **kw) as ctx:
        ctx.submit_host(text, spans_of(off, ln))
        d = (ctx.diag(len(seqs)), ctx.diag_reverse(len(seqs))) if diag else None
        table = ctx.finish_dict()
        stats = ctx.stats()
    return table, d, stats


def assert_diag_equal(got, want):
    for f in want.dtype.names:
        assert (got[f] == want[f]).all(), (f, np.nonzero(got[f] != want[f])[0][:5])


def check(seqs, adapters, diag=False, cells=True, **kw):
    want = expected(seqs, adapters, **kw)
    table, d, st = gpu_run(seqs, adapters, diag=diag, **kw)
    assert table == want["table"]
    assert st["counted"] == want["counted"]
    assert st["reverse_reads"] == want["reverse_reads"]
    assert st["reverse_counted"] == want["reverse_counted"]
    if cells:
        assert st["dp_cells"] == want["cells"]
    if diag:
        assert_diag_equal(d[0], want["fdiag"])
        assert_diag_equal(d[1], want["rdiag"])
    return want, st


@pytest.mark.parametrize("mode", ["windowed", "full", "diagnostics", "skip_translation"])
def test_mixed_strands(mode):
    rng = random.Random(101)
    seqs = make_reads(rng, PREFIX, SUFFIX, 6000, alphabet=b"ACGTacgtUuN-", empty=0.02)
    # non-ASCII bytes: X for translation; with skip_translation nearly every such region is invalid UTF-8 (reversal
    # breaks the multi-byte sequences up), so these reads are dropped on both strands
    seqs += make_reads(rng, PREFIX, SUFFIX, 1000, alphabet=b"ACGTN" + ODD)
    kw = {"windowed": dict(dp_compute_all=True), "full": dict(dp_mode=1, dp_compute_all=True),
          "diagnostics": dict(diag=True), "skip_translation": dict(skip_translation=True, dp_compute_all=True)}[mode]
    want, st = check(seqs, (PREFIX, SUFFIX), **kw)
    assert want["reverse_counted"] > 500


def test_default_path_without_compute_all():
    # the suffix alignments of prefix-rejected reads are skipped (fewer cells), the tables are the same
    rng = random.Random(102)
    seqs = make_reads(rng, PREFIX, SUFFIX, 5000)
    check(seqs, (PREFIX, SUFFIX), cells=False)
    check(seqs, (PREFIX, SUFFIX), cells=False, dp_mode=1)


@pytest.mark.parametrize("A", [8, 12, 14, 20, 33, 48, 64])
def test_adapter_lengths(A):
    rng = random.Random(200 + A)
    pre = bytes(rng.choice(b"ACGT") for _ in range(A))
    suf = bytes(rng.choice(b"ACGT") for _ in range(A))
    seqs = make_reads(rng, pre, suf, 3000)
    check(seqs, (pre, suf), dp_compute_all=True)


def test_general_scan_and_diagnostics():
    rng = random.Random(103)
    seqs = make_reads(rng, PREFIX, SUFFIX, 3000, alphabet=b"ACGTacgtUN", empty=0.02)
    check(seqs, (PREFIX, SUFFIX), dp_compute_all=True, force_general_scan=True)
    check(seqs, (PREFIX, SUFFIX), diag=True, force_general_scan=True)


def test_small_batches_alternate_lanes():
    rng = random.Random(104)
    seqs = make_reads(rng, PREFIX, SUFFIX, 7000, empty=0.05)
    check(seqs, (PREFIX, SUFFIX), dp_compute_all=True, batch_reads=97)
    check(seqs, (PREFIX, SUFFIX), cells=False, batch_reads=64, skip_translation=True)


def test_all_empty_and_all_forward_batches():
    rng = random.Random(105)
    fwd = [s for s in make_reads(rng, PREFIX, SUFFIX, 2000) if s]
    seqs = [b""] * 64 + fwd[:64] + [b""] * 64 + [strand_oracle.revcomp(s) for s in fwd[64:128]]
    check(seqs, (PREFIX, SUFFIX), dp_compute_all=True, batch_reads=64)
    check(seqs, (PREFIX, SUFFIX), diag=True)


def test_profiling_covers_both_passes():
    rng = random.Random(106)
    seqs = make_reads(rng, PREFIX, SUFFIX, 4000)
    text, off, ln = oracle.pack_reads(seqs)
    want = expected(seqs, (PREFIX, SUFFIX))
    with api.Context((PREFIX, SUFFIX), both_strands=True, batch_reads=500) as ctx:
        ctx.set_profiling(True)
        ctx.submit_host(text, spans_of(off, ln))
        assert ctx.finish_dict() == want["table"]
        st = ctx.stats()
    assert st["ms_total"] > 0 and st["ms_scan"] > 0 and st["reverse_counted"] == want["reverse_counted"]


def test_two_contexts_merged():
    torch = pytest.importorskip("torch")
    rng = random.Random(107)
    seqs = make_reads(rng, PREFIX, SUFFIX, 6000)
    want = expected(seqs, (PREFIX, SUFFIX))
    halves = [seqs[:2500], seqs[2500:]]
    ctxs = [api.Context((PREFIX, SUFFIX), both_strands=True) for _ in halves]
    try:
        for ctx, part in zip(ctxs, halves):
            text, off, ln = oracle.pack_reads(part)
            ctx.submit_host(text, spans_of(off, ln))
        sizes = ctxs[1].partition_sizes(1)
        buf = torch.empty(int(sizes[0]), dtype=torch.uint8, device="cuda")
        ctxs[1].partition_fill(1, buf.data_ptr(), [0])
        st = [c.stats() for c in ctxs]
        ctxs[0].absorb(buf.data_ptr(), sizes[0])
        assert ctxs[0].finish_dict() == want["table"]
        assert sum(s["reverse_reads"] for s in st) == want["reverse_reads"]
        assert sum(s["reverse_counted"] for s in st) == want["reverse_counted"]
    finally:
        for c in ctxs:
            c.close()
    with api.MultiContext((PREFIX, SUFFIX), devices=[0], both_strands=True) as m:
        text, off, ln = oracle.pack_reads(seqs)
        m.contexts[0].submit_host(text, spans_of(off, ln))
        assert m.finish_dict() == want["table"]
        ms = m.stats()
    assert ms["reverse_reads"] == want["reverse_reads"] and ms["reverse_counted"] == want["reverse_counted"]


@pytest.mark.parametrize("gz", [True, False])
def test_run_file(tmp_path, gz):
    rng = random.Random(108)
    seqs = [s for s in make_reads(rng, PREFIX, SUFFIX, 5000) if s]
    fq = b"".join(b"@r%d\n%s\n+\n%s\n" % (i, s, b"F" * len(s)) for i, s in enumerate(seqs))
    path = tmp_path / ("r.fq.gz" if gz else "r.fq")
    path.write_bytes(gzip.compress(fq) if gz else fq)
    want = expected(seqs, (PREFIX, SUFFIX))
    with api.Context((PREFIX, SUFFIX), both_strands=True) as ctx:
        assert ctx.run_file(str(path), allow_text=not gz) == len(seqs)
        assert ctx.finish_dict() == want["table"]
        st = ctx.stats()
    assert st["reverse_reads"] == want["reverse_reads"] and st["reverse_counted"] == want["reverse_counted"]
    out = api.find_variants(str(path), (PREFIX.decode(), SUFFIX.decode()), show_progress=False, allow_text=not gz,
                            both_strands=True)
    cols = out.to_pydict() if hasattr(out, "to_pydict") else out.to_dict(as_series=False)
    assert {k.encode(): v for k, v in zip(cols["sequence"], cols["count"])} == want["table"]


def test_read_diagnostics_columns():
    fwd = PREFIX + b"ATGGCTAGCAAAGGAGAAGAA" + SUFFIX
    seqs = [fwd, strand_oracle.revcomp(fwd), b"", b"ACGTACGT"]
    t = api.read_diagnostics(seqs, (PREFIX, SUFFIX), both_strands=True).to_pydict()
    assert t["strand"] == [1, -1, None, None]
    assert t["region"] == [b"ATGGCTAGCAAAGGAGAAGAA", b"ATGGCTAGCAAAGGAGAAGAA", None, None]
    assert t["rev_start"][0] is None and t["rev_start"][1] == len(PREFIX) and t["rev_start"][2] is None
    assert t["rev_exact_prefix"][3] is None and t["rev_score_prefix"][3] is not None
    assert t["start"][1] is None
    plain = api.read_diagnostics(seqs, (PREFIX, SUFFIX)).to_pydict()
    assert "strand" not in plain and plain["region"] == [b"ATGGCTAGCAAAGGAGAAGAA", None, None, None]


def test_submit_device_overlapping_spans_beyond_4gib():
    # 4.4 M spans of 1000 bases over 64 distinct reverse-complemented reads: every read is retried and the gathered
    # text would exceed 32-bit offsets, so the call is cut into smaller batches
    torch = pytest.importorskip("torch")
    rng = random.Random(109)
    variants = [bytes(rng.choice(b"ACGT") for _ in range(30)) for _ in range(64)]
    distinct = []
    for v in variants:
        body = PREFIX + v + SUFFIX
        pad = 1000 - len(body)
        distinct.append(strand_oracle.revcomp(bytes(rng.choice(b"ACGT") for _ in range(pad // 2)) + body +
                                       bytes(rng.choice(b"ACGT") for _ in range(pad - pad // 2))))
    text, off, ln = oracle.pack_reads(distinct)
    n = 4_400_000
    pick = np.random.default_rng(5).integers(0, 64, n)
    assert int(ln[pick].astype(np.int64).sum()) > 2 ** 32
    mult = np.bincount(pick, minlength=64)
    want = {}
    p = oracle.make_params((PREFIX, SUFFIX))
    for i in range(64):
        t, o, l = oracle.pack_reads([distinct[i]])
        for k, v in strand_oracle.process_reads_both_strands(p, t, o, l)[0].items():
            want[k] = want.get(k, 0) + v * int(mult[i])
    d_text = torch.from_numpy(text.copy()).cuda()
    sp = np.stack([off[pick], ln[pick]], 1).astype(np.uint32)
    d_sp = torch.from_numpy(sp.view(np.int32).copy()).cuda()
    with api.Context((PREFIX, SUFFIX), both_strands=True, batch_reads=n) as ctx:
        ctx.submit_device(d_text.data_ptr(), d_text.numel(), d_sp.data_ptr(), n)
        got = ctx.finish_dict()
        st = ctx.stats()
    assert got == want
    assert st["reverse_reads"] == n and st["reverse_counted"] == sum(want.values())
