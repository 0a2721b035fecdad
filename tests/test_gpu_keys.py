"""The key and count path (csrc/kernels_count.cu) at every key length, against the oracle and the host hash.

A batch that meets an empty table builds its keys with k3_keys_tile and inserts them with k4_insert / k4_publish;
every later batch runs k34_keys_count, which translates with its own loop and probes the table itself: keys whose
padded length fits K34_ROW_BYTES take the piped probe (home slot only), longer ones k34_probe (up to K34_PROBES
slots).  Both kernels must produce the same bytes and the same hash, or a later batch misses the row an earlier one
made and the table gets a second row for one key.  The tests here send keys of 1 to 5000 bytes through both kernels
(one batch, and batches of 97 and 1000 reads on two lanes), near-identical keys under forced hash collisions, and
compare every hash the device stored with api.hash_key (the host reference that test_keys_cpu.py pins).

Reads are lead + PREFIX + region + SUFFIX + tail with exact adapters: the alignment is not under test here.
"""
import collections
import random
import struct

import numpy as np
import pytest
import torch

import oracle
from vfind_b200 import api

pytestmark = pytest.mark.gpu

PREFIX = b"GGGCCCAGCCGGCCGGAT"
SUFFIX = b"CCGGAGGCGGAGGTTCAG"
HINT = 1 << 18                       # table_capacity_hint -> 2^19 slots (table_init), never outgrown here
SLOTS = 1 << 19
MAGIC = 0x5646423230304B31
BIG_COUNTS = (2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 40 + 3)
BATCHINGS = (None, 97, 1000)         # None: all reads in one batch

CANON = b"ACGT"
RAW = bytes(range(0x21, 0x7F))
# one byte the arithmetic translate must hand to the per-byte tables (N, '-', >= 0x80), or that it must fold
# (lower case, U)
ODD = [b"N", b"n", b"a", b"c", b"g", b"t", b"u", b"U", b"-", b"\x80", b"\xc3", b"\xff"]
AA_OF = None


def a16(x):
    return (x + 15) & ~15


def aa_of(codon):
    global AA_OF
    if AA_OF is None:
        AA_OF = {bytes(c): oracle.translate(bytes(c)) for c in
                 (bytes((x, y, z)) for x in CANON for y in CANON for z in CANON)}
    return AA_OF[codon]


def key_of(region, translated):
    if translated:
        return oracle.translate(region)
    return region if oracle.is_utf8(region) else None


# ---------------------------------------------------------------------------------------------------- read sets
def rand_region(rng, n, translated):
    return bytes(rng.choice(CANON if translated else RAW) for _ in range(3 * n if translated else n))


def change_unit(rng, region, j, translated):
    """The region with key byte j replaced by a different one (codon j, for translated keys)."""
    if translated:
        old = aa_of(region[3 * j:3 * j + 3])
        while True:
            c = bytes(rng.choice(CANON) for _ in range(3))
            if aa_of(c) != old:
                return region[:3 * j] + c + region[3 * j + 3:]
    b = rng.choice([x for x in RAW if x != region[j]])
    return region[:j] + bytes([b]) + region[j + 1:]


def family(rng, base, n, translated):
    """Keys equal to the base's but in one byte (the last, the first, 79 / 80 / 81, 511 / 512, four in the final
    padded chunk) or one byte shorter or longer."""
    out = [change_unit(rng, base, j, translated) for j in sorted({n - 1, 0, 79, 80, 81, 511, 512}) if j < n]
    out += [change_unit(rng, base, rng.randrange(16 * ((n - 1) // 16), n), translated) for _ in range(4)]
    unit = 3 if translated else 1
    if n > 1:
        out.append(base[:-unit])
    out.append(base + rand_region(rng, 1, translated))
    return out


def odd_bytes(base, n):
    """An odd byte at each of the twelve positions of a translate group: the first group, one in the middle, the
    last (possibly partial) one and one past key word 128."""
    groups = {0, (n - 1) // 4 // 2, (n - 1) // 4}
    if n > 4 * 128:
        groups |= {128, 129}
    for g in sorted(groups):
        for j in range(12):
            pos = 12 * g + j
            if pos < 3 * n:
                yield base[:pos] + ODD[(g + j) % 12] + base[pos + 1:]


def utf8_cases(rng, n):
    """Raw keys with multi-byte characters (kept) and with invalid UTF-8 (dropped), n bytes long."""
    if n < 6:
        return []
    body = lambda k: rand_region(rng, k, False)
    return [body(n - 5) + "é€".encode(), "€".encode() + body(n - 3),
            body(n - 1) + b"\xff", body(n - 1) + b"\xc3", body(n - 3) + b"\xed\xa0\x80", b"\x80" + body(n - 1)]


def regions_for(rng, lengths, per_len, translated, families=True):
    regions = []
    for n in lengths:
        fresh = [rand_region(rng, n, translated) for _ in range(per_len)]
        regions += fresh
        if not families:
            continue
        regions += family(rng, fresh[0], n, translated)
        if translated:
            regions += list(odd_bytes(fresh[1], n))
            regions += [fresh[2] + b"A", fresh[2] + b"GC"]          # 3k+1 and 3k+2 bases: no key
        else:
            regions += utf8_cases(rng, n)
    return regions


def distinct_home_slots(regions, translated):
    """Drop the regions whose key would share its home slot with another key: the piped probe looks at the home
    slot only, so a second key there is counted by the insert kernels and not by the fused kernel."""
    taken, out = {}, []
    for r in regions:
        k = key_of(r, translated)
        if k is not None:
            s = api.hash_key(k) & (SLOTS - 1)
            if taken.setdefault(s, k) != k:
                continue
        out.append(r)
    return out


class ReadSet:
    def __init__(self, name, translated, regions, seed, home_slots=True):
        rng = random.Random(seed)
        self.name, self.translated = name, translated
        if home_slots:
            regions = distinct_home_slots(regions, translated)
        reads = []
        for r in regions:
            for _ in range(rng.randint(1, 3)):
                lead = bytes(rng.choice(CANON) for _ in range(rng.randrange(8)))
                tail = bytes(rng.choice(CANON) for _ in range(rng.randrange(8)))
                reads.append(lead + PREFIX + r + SUFFIX + tail)
        rng.shuffle(reads)
        self.reads = reads
        self.text, off, ln = oracle.pack_reads(reads)
        self.spans = np.zeros(len(reads), dtype=api.SPAN_DTYPE)
        self.spans["off"], self.spans["len"] = off, ln
        p = oracle.make_params((PREFIX, SUFFIX), skip_translation=not translated)
        self.want = oracle.process_reads(p, self.text, off, ln, n_threads=8)[0]
        # the oracle finds exactly the regions that were built (the adapters are exact), so the key lengths are the
        # ones this set is meant to reach
        expect = collections.Counter()
        for rd in reads:
            k = key_of(rd[rd.index(PREFIX) + len(PREFIX):rd.rindex(SUFFIX)], translated)
            if k is not None:
                expect[k] += 1
        assert self.want == dict(expect), name
        self.counted = sum(self.want.values())


def _classes():
    """name -> (translated, lengths, keys per length, families)."""
    c = {}
    for lens, per in (((range(1, 21)), 12), ((31, 32, 33), 40), ((63, 64, 65, 66, 67), 30), ((79, 80), 60),
                      ((81, 95, 96, 97), 30), ((127, 128, 129), 30), ((255, 256, 257), 25), ((511, 512, 513, 514), 12),
                      ((1023, 1024, 1025), 10), ((1500,), 16)):
        c["aa_" + "_".join(map(str, sorted({min(lens), max(lens)})))] = (True, tuple(lens), per, True)
    for lens, per in (((range(1, 49)), 6), ((63, 64, 65), 40), ((79, 80), 60), ((81, 95, 96, 97), 30),
                      ((127, 128, 129), 30), ((511, 512, 513), 16), ((1023, 1024, 1025), 12), ((2047, 2048, 2049), 8),
                      ((4095, 4096, 4097), 6), ((4999, 5000, 5003), 6)):
        c["raw_" + "_".join(map(str, sorted({min(lens), max(lens)})))] = (False, tuple(lens), per, True)
    return c


CLASSES = _classes()
MIXES = ("aa_short_rare_long", "aa_long_rare_short", "raw_short_rare_long", "raw_long_rare_short")
_sets = {}


def read_set(name):
    if name in _sets:
        return _sets[name]
    seed = sum(name.encode()) * 7919 + len(name)
    rng = random.Random(seed)
    if name in CLASSES:
        translated, lens, per, fam = CLASSES[name]
        regions = regions_for(rng, lens, per, translated, fam)
    else:
        translated = name.startswith("aa")
        # the key block of k34_keys_count is sized from the batch's average span: a rare long key in a batch of
        # short ones does not fit it, a rare short one in a batch of long ones leaves it mostly empty
        short, long_ = ((7, 8, 9, 10), (1500,)) if translated else ((21, 24, 30), (4097,))
        if name.endswith("short_rare_long"):
            regions = regions_for(rng, short, 250, translated, False) + regions_for(rng, long_, 6, translated, False)
        else:
            mid = (255, 256, 257) if translated else (511, 512, 513)
            regions = regions_for(rng, mid, 70, translated, False) + regions_for(rng, (1, 2, 3), 2, translated, False)
    _sets[name] = ReadSet(name, translated, regions, seed)
    return _sets[name]


# ---------------------------------------------------------------------------------------------------- helpers
def context(batch_reads, n_reads, **kw):
    return api.Context((PREFIX, SUFFIX), skip_translation=kw.pop("skip_translation"), batch_reads=batch_reads or n_reads,
                       table_capacity_hint=HINT, **kw)


def table_of(ctx):
    """The table from the raw columns of finish_arrays, with the checks a dict would hide: no key twice, one row per
    table row, counts that add up to what was counted."""
    offsets, data, counts = ctx.finish_arrays()
    st = ctx.stats()
    assert offsets.dtype == np.uint64 and counts.dtype == np.uint64
    assert int(offsets[0]) == 0 and int(offsets[-1]) == len(data) and (np.diff(offsets.astype(np.int64)) > 0).all()
    raw = data.tobytes()
    keys = [raw[int(offsets[i]):int(offsets[i + 1])] for i in range(len(counts))]
    assert len(set(keys)) == len(keys), "a key has two rows"
    assert len(keys) == st["unique"]
    assert sum(int(c) for c in counts) == st["counted"]
    return dict(zip(keys, (int(c) for c in counts))), st


def arrow_table(ctx):
    import pyarrow as pa
    batch = ctx.finish_arrow()
    assert batch.schema.field("count").type == pa.uint64()
    keys = [s.encode() for s in batch.column(0).to_pylist()]
    assert len(set(keys)) == len(keys)
    return dict(zip(keys, batch.column(1).to_pylist()))


def times(table, k):
    return {key: k * v for key, v in table.items()}


def two_passes(rs, batch_reads, **kw):
    """The reads twice into one context: (table after pass 1, stats, table after pass 2, stats, context)."""
    ctx = context(batch_reads, len(rs.reads), skip_translation=not rs.translated, **kw)
    ctx.submit_host(rs.text, rs.spans)
    t1, s1 = table_of(ctx)
    ctx.submit_host(rs.text, rs.spans)
    t2, s2 = table_of(ctx)
    return t1, s1, t2, s2, ctx


def n_batches(n, batch_reads):
    return 1 if batch_reads is None else (n + batch_reads - 1) // batch_reads


def parse_chunk(raw):
    """Rows (hash, count, key) of one chunk (csrc/vfb_internal.cuh: ChunkHeader, then hashes, counts, key offsets,
    lengths and the 16-byte padded keys), after checking its layout; the padding of every key must be zero."""
    magic, n, kb, _ = struct.unpack_from("<4Q", raw, 0)
    assert magic == MAGIC
    assert len(raw) == 32 + 3 * a16(8 * n) + a16(4 * n) + a16(kb)
    o = 32
    hashes = np.frombuffer(raw, np.uint64, n, o); o += a16(8 * n)
    counts = np.frombuffer(raw, np.uint64, n, o); o += a16(8 * n)
    koff = np.frombuffer(raw, np.uint64, n, o); o += a16(8 * n)
    klen = np.frombuffer(raw, np.uint32, n, o); o += a16(4 * n)
    assert sum(a16(int(x)) for x in klen) == kb
    spans = sorted((int(koff[i]), a16(int(klen[i]))) for i in range(n))
    assert all(a + b <= c for (a, b), (c, _) in zip(spans, spans[1:]))          # keys do not overlap
    rows = []
    for i in range(n):
        k0, kl = o + int(koff[i]), int(klen[i])
        assert raw[k0 + kl:k0 + a16(kl)] == b"\0" * (a16(kl) - kl), "non-zero key padding"
        rows.append((int(hashes[i]), int(counts[i]), raw[k0:k0 + kl]))
    return rows


def export(ctx, n_parts):
    """partition_sizes / partition_fill into a buffer filled with 0xA5 (bytes the fill does not write show):
    (device buffer, offsets, sizes, host bytes of each chunk)."""
    sizes = ctx.partition_sizes(n_parts)
    offs = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64)
    buf = torch.full((int(sum(sizes)),), 0xA5, dtype=torch.uint8, device="cuda")
    ctx.partition_fill(n_parts, buf.data_ptr(), offs)
    host = buf.cpu().numpy().tobytes()
    return buf, offs, sizes, [host[int(offs[p]):int(offs[p]) + sizes[p]] for p in range(n_parts)]


# ---------------------------------------------------------------------------------------------------- tests
ALL = list(CLASSES) + list(MIXES)


@pytest.mark.parametrize("name", ALL)
def test_both_key_kernels_count_every_length(name, monkeypatch):
    """Each read set in one batch and in batches of 97 and 1000 reads, twice into the same context: the table is the
    oracle's, then twice the oracle's.  The first batch of a context builds its keys with k3_keys_tile, every later
    one with k34_keys_count; on the second pass every key already has a row, so the fused kernel must find each one
    itself (piped compare or k34_probe, its own hash): its hits grow by exactly the reads counted."""
    rs = read_set(name)
    n = len(rs.reads)
    for br in BATCHINGS:
        t1, s1, t2, s2, ctx = two_passes(rs, br)
        ctx.close()
        nb = n_batches(n, br)
        assert t1 == rs.want, (name, br)
        assert t2 == times(rs.want, 2), (name, br)
        assert s1["counted"] == rs.counted and s2["unique"] == len(rs.want)
        assert s1["fused_batches"] == nb - 1 and s2["fused_batches"] == 2 * nb - 1, (name, br)
        assert s2["fused_hits"] - s1["fused_hits"] == rs.counted, (name, br, "the fused kernel missed existing rows")
    monkeypatch.setenv("VFB_FUSED_COUNT", "0")
    t1, s1, t2, s2, ctx = two_passes(rs, 97)
    ctx.close()
    assert t1 == rs.want and t2 == times(rs.want, 2)
    assert s2["fused_batches"] == 0 and s2["fused_hits"] == 0


def collision_set(translated, n, tail_only):
    """Eight keys of n bytes with their families; tail_only: forty keys that share everything but the final padded
    chunk (whichever of them holds a home slot, the others of its hash bit meet it there)."""
    name = "collide_%s_%d%s" % ("aa" if translated else "raw", n, "_tail" if tail_only else "")
    if name in _sets:
        return _sets[name]
    rng = random.Random(name)
    regions = []
    if tail_only:
        head = rand_region(rng, 16 * ((n - 1) // 16), translated)
        regions = [head + rand_region(rng, n - 16 * ((n - 1) // 16), translated) for _ in range(40)]
    else:
        for _ in range(8):
            base = rand_region(rng, n, translated)
            regions += [base] + family(rng, base, n, translated)
    _sets[name] = ReadSet(name, translated, regions, n, home_slots=False)
    return _sets[name]


COLLIDE = [(True, n, False) for n in (20, 80, 81, 129, 513, 1025)] + \
          [(False, n, False) for n in (16, 80, 81, 97, 513, 1025, 4097)] + \
          [(t, n, True) for t in (True, False) for n in (80, 81)]


@pytest.mark.parametrize("bits", [1, 9])
@pytest.mark.parametrize("translated,n,tail_only", COLLIDE,
                         ids=["%s%d%s" % ("aa" if t else "raw", n, "tail" if o else "") for t, n, o in COLLIDE])
def test_near_identical_keys_under_forced_collisions(translated, n, tail_only, bits, monkeypatch):
    """Keys that differ from one another in a single byte (first, last, 79-81, 511 / 512, final padded chunk) or in
    length, all hashed to 1 or 9 bits: every probe meets rows with the same tag and must decide on the bytes."""
    rs = collision_set(translated, n, tail_only)
    for fused in ("1", "0"):
        monkeypatch.setenv("VFB_FUSED_COUNT", fused)
        for br in BATCHINGS:
            t1, s1, t2, s2, ctx = two_passes(rs, br, debug_hash_bits=bits)
            ctx.close()
            assert t1 == rs.want and t2 == times(rs.want, 2), (fused, br)
            assert s2["counted"] == 2 * rs.counted
            assert (s2["fused_batches"] > 0) == (fused == "1")


@pytest.mark.parametrize("name", ALL)
def test_device_hashes_equal_the_host_reference(name):
    """Every row of the table, exported as 1, 7 and 64 chunks: the stored hash is api.hash_key of the key bytes, the
    row sits in the chunk of its owner, the key's padding is zero, the chunks are disjoint and together are the
    table.  Rows come from both kernels (batches of 97: k3_keys_tile makes the first batch's rows, k34_keys_count the
    rest)."""
    rs = read_set(name)
    t1, s1, t2, s2, ctx = two_passes(rs, 97)
    with ctx:
        assert s2["fused_batches"] > 0
        for n_parts in (1, 7, 64):
            _, _, _, chunks = export(ctx, n_parts)
            seen = {}
            for p, raw in enumerate(chunks):
                for h, c, k in parse_chunk(raw):
                    assert h == api.hash_key(k), (name, len(k))
                    assert api.key_owner(h, n_parts) == p
                    assert k not in seen
                    seen[k] = c
            assert seen == t2


@pytest.mark.parametrize("name", ALL)
def test_absorb_long_keys_and_64_bit_counts(name):
    """Chunks absorbed twice double the counts; counts patched to values at and past 2^32 add up exactly in a fresh
    context and in one that already holds keys from reads; reads submitted afterwards are counted by the fused kernel
    against the rows absorb made."""
    rs = read_set(name)
    n = len(rs.reads)
    skip = not rs.translated
    with context(None, n, skip_translation=skip) as src:
        src.submit_host(rs.text, rs.spans)
        buf, offs, sizes, chunks = export(src, 7)
    with context(None, n, skip_translation=skip) as dst:
        for _ in range(2):
            for p in range(7):
                dst.absorb(buf.data_ptr() + int(offs[p]), sizes[p])
        got, st = table_of(dst)
        assert got == times(rs.want, 2) and st["counted"] == 2 * rs.counted
    # the chunk with the most rows, its counts replaced
    p = max(range(7), key=lambda q: len(parse_chunk(chunks[q])))
    raw = bytearray(chunks[p])
    rows = struct.unpack_from("<Q", raw, 8)[0]
    big = np.array([BIG_COUNTS[i % len(BIG_COUNTS)] for i in range(rows)], dtype=np.uint64)
    raw[32 + a16(8 * rows):32 + a16(8 * rows) + 8 * rows] = big.tobytes()
    patched = {k: c for _, c, k in parse_chunk(bytes(raw))}
    dev = torch.frombuffer(raw, dtype=torch.uint8).cuda()
    half = n // 2
    before = collections.Counter()
    for rd in rs.reads[:half]:
        k = key_of(rd[rd.index(PREFIX) + len(PREFIX):rd.rindex(SUFFIX)], rs.translated)
        if k is not None:
            before[k] += 1
    for pre_reads in (0, half):
        with context(None, n, skip_translation=skip) as ctx:
            if pre_reads:
                ctx.submit_host(rs.text, rs.spans[:pre_reads].copy())
            want = collections.Counter(before if pre_reads else {})
            for _ in range(2):
                ctx.absorb(dev.data_ptr(), len(raw))
                want.update(patched)
            got, st = table_of(ctx)
            assert got == dict(want) and arrow_table(ctx) == dict(want)
            assert st["counted"] == sum(want.values())
            known = set(want)
            s0 = st
            ctx.submit_host(rs.text, rs.spans)
            want.update(rs.want)
            got, st = table_of(ctx)
            assert got == dict(want) and arrow_table(ctx) == dict(want)
            assert st["fused_batches"] - s0["fused_batches"] == 1
            # one batch: exactly the reads whose key had a row before it are counted by the fused kernel
            assert st["fused_hits"] - s0["fused_hits"] == sum(c for k, c in rs.want.items() if k in known)


def test_empty_parts_are_chunks_of_zero_rows():
    """partition_sizes counts a 32-byte chunk for a part without rows (an empty table has only such parts): the fill
    must write its header, so that absorbing it adds nothing instead of failing on whatever the buffer held."""
    rs = read_set("raw_4999_5003")
    one = next(i for i, rd in enumerate(rs.reads) if key_of(rd[rd.index(PREFIX) + len(PREFIX):rd.rindex(SUFFIX)], False))
    for n_reads in (0, 1):
        with context(None, 1, skip_translation=True) as src:
            if n_reads:
                src.submit_host(rs.text, rs.spans[one:one + 1].copy())
            want = src.finish_dict()
            _, _, sizes, chunks = export(src, 64)
        assert sorted(sizes)[:63] == [32] * 63
        got = {}
        for raw in chunks:
            rows = parse_chunk(raw)
            assert len(raw) > 32 or rows == []
            with context(None, 1, skip_translation=True) as dst:
                dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
                dst.absorb(dev.data_ptr(), len(raw))
                got.update(dst.finish_dict())
        assert got == want and len(want) == n_reads
