"""CPU tests of the shipped library: it loads, exports every symbol include/vfind_b200.h
declares, keeps the reference's signature, and refuses to compute without a GPU."""
import ctypes
import inspect
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from vfind_b200 import build
    build.build()
    from vfind_b200 import api
    return api.load_library()


def test_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "vfind_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(vfb_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 25
    for n in sorted(names):
        assert hasattr(lib, n), n
    assert lib.vfb_abi_version() == 1


def test_struct_layouts_match_header(lib):
    from vfind_b200 import api
    p = api.Params()
    lib.vfb_default_params(ctypes.byref(p))
    assert p.struct_size == ctypes.sizeof(api.Params)
    assert (p.match_score, p.mismatch_score, p.gap_open_penalty, p.gap_extend_penalty) == (3, -2, 5, 2)
    assert (p.accept_prefix_alignment, p.accept_suffix_alignment) == (0.75, 0.75)
    assert (p.n_threads, p.queue_len, p.skip_translation, p.show_progress, p.device) == (3, 2, 0, 1, -1)
    assert api.DIAG_DTYPE.itemsize == 32 and api.SPAN_DTYPE.itemsize == 8


def test_signature_matches_reference(golden):
    from vfind_b200 import find_variants
    import vfind
    assert vfind.find_variants is find_variants
    sig = inspect.signature(find_variants)
    positional = [n for n, p in sig.parameters.items() if p.kind == p.POSITIONAL_OR_KEYWORD]
    assert positional == golden["signature_order"]                       # src/lib.rs:169-182
    for k, v in golden["signature_defaults"].items():
        assert sig.parameters[k].default == v, k
    extras = [n for n, p in sig.parameters.items() if p.kind == p.KEYWORD_ONLY]
    assert extras and all(sig.parameters[n].default is not inspect.Parameter.empty for n in extras)


def test_argument_coercion_errors(tmp_path):
    from vfind_b200 import find_variants
    ad = ("ACGT", "TTGA")
    with pytest.raises(FileNotFoundError):
        find_variants(str(tmp_path / "nope.fq.gz"), ad)
    f = tmp_path / "x.fq.gz"
    f.write_bytes(b"")
    with pytest.raises(TypeError):
        find_variants(123, ad)
    with pytest.raises(TypeError):
        find_variants(str(f), "ACGT")
    with pytest.raises(ValueError):
        find_variants(str(f), ("A", "C", "G"))
    with pytest.raises(TypeError):
        find_variants(str(f), ad, match_score=3.5)
    with pytest.raises(OverflowError):
        find_variants(str(f), ad, match_score=2 ** 31)
    with pytest.raises(OverflowError):
        find_variants(str(f), ad, n_threads=-1)
    with pytest.raises(TypeError):
        find_variants(str(f), ad, skip_translation="yes")


def test_threshold_validation_precedes_device_use(lib, golden):
    # src/lib.rs:100-110 — the message and exception type are the reference's
    from vfind_b200 import api
    for thr in (0.0, -1.0, 1.01, float("nan")):
        with pytest.raises(ValueError, match=golden["threshold_error"]):
            api.Context(("ACGT", "TTGA"), accept_prefix_alignment=thr)
        with pytest.raises(ValueError, match=golden["threshold_error"]):
            api.Context(("ACGT", "TTGA"), accept_suffix_alignment=thr)


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from vfind_b200 import api
    with pytest.raises(RuntimeError, match="no CUDA device"):
        api.Context(("ACGT", "TTGA"))


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "vfind_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
                assert "vfind_oracle.h" not in src and "libvfind_oracle" not in src, f


def test_synth_host_is_deterministic_and_shaped(lib):
    from vfind_b200 import api
    cfg = api.synth_cfg(seed=7, read_len=150, adapter_len=20, region_len=99, n_variants=50, p_err=0.3)
    pre, suf = api.synth_adapters(cfg)
    assert len(pre) == len(suf) == 20 and pre != suf
    t1, s1 = api.synth_host(cfg, 0, 300)
    t2, s2 = api.synth_host(cfg, 100, 50)
    assert t1.size == 300 * 150 and (s1["len"] == 150).all()
    assert (t1[100 * 150:150 * 150] == t2).all()             # any shard reproduces the stream
    assert set(np.unique(t1)) <= set(b"ACGTN")
    reads = [t1[i * 150:(i + 1) * 150].tobytes() for i in range(300)]
    exact = sum(1 for r in reads if pre in r and suf in r)
    assert 100 < exact < 200                                  # ~ (1-0.3)^2 of reads are exact/exact


def test_hash_reference_properties(lib):
    # the host twin of the device hash (hash.h) is restated in test_keys_cpu.py and compared with
    # every hash the device stores in test_gpu_keys.py; here: chunk header rejects garbage
    from vfind_b200 import api
    rows = ctypes.c_uint64(0)
    buf = np.zeros(64, dtype=np.uint8)
    assert lib.vfb_chunk_rows(buf.ctypes.data, 64, ctypes.byref(rows)) == api.VFB_ERR_FORMAT


def test_oracle_side_generator_matches_the_library(lib, tmp_path):
    """bench.py --impl reference takes its inputs from oracle/synth_host.c (it must not load the product): the two
    generators compile the same header and must produce the same bytes; the FASTQ writer frames them as records."""
    import gzip
    import oracle
    from vfind_b200 import api
    for kw in (dict(), dict(seed=5, read_len=300, adapter_len=40, region_len=210, p_err=0.15, force_indel=0),
               dict(seed=9, read_len=150, adapter_len=20, region_len=99, n_variants=1000, zipf=0, noise=0.0)):
        cfg = api.synth_cfg(**kw)
        ocfg = oracle.synth_cfg(**kw)
        assert bytes(cfg) == bytes(ocfg)
        t1, s1 = api.synth_host(cfg, 12345, 3000)
        t2, off, ln = oracle.synth_reads(ocfg, 12345, 3000, 3)
        assert (t1 == t2).all() and (off == s1["off"]).all() and (ln == s1["len"]).all()
        assert oracle.synth_adapters(ocfg) == api.synth_adapters(cfg)
    cfg = oracle.synth_cfg()
    p = str(tmp_path / "s.fq.gz")
    tb, fb = oracle.write_fastq(cfg, 7, 2000, p, bgzf=True, threads=3)
    raw = gzip.open(p).read()
    text, _, _ = oracle.synth_reads(cfg, 7, 2000)
    L = cfg.read_len
    assert tb == len(raw) == 2000 * (2 * L + 17) and fb == os.path.getsize(p)
    for i in (0, 1, 1999):
        rec = raw[i * (2 * L + 17):(i + 1) * (2 * L + 17)].split(b"\n")
        assert rec[0] == b"@r%010d" % (7 + i) and rec[1] == text[i * L:(i + 1) * L].tobytes() and rec[2] == b"+" and rec[3] == b"F" * L


def test_translate_fast_path_arithmetic(lib):
    """The key kernel's arithmetic translate (csrc/translate_fast.h, host build of the same code): twelve bases ->
    four amino acids whenever all twelve are canonical; anything else must be flagged (the kernel then takes the
    per-byte tables).  Against the oracle's translate (src/lib.rs:16-44, tables :52-95)."""
    import ctypes as C
    import itertools
    import random

    import oracle

    fn = lib.vfb_debug_translate12
    fn.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_int)]
    fn.restype = C.c_int
    canonical = b"ACGTUacgtu"

    def run(b12):
        out = C.create_string_buffer(4)
        ok = C.c_int(-1)
        assert fn(bytes(b12), out, C.byref(ok)) == 0
        return out.raw, ok.value

    # every canonical triplet in each of the four codon slots, the other slots filled with a varying background
    rng = random.Random(5)
    for trip in itertools.product(canonical, repeat=3):
        for slot in range(4):
            b = bytearray(rng.choice(canonical) for _ in range(12))
            b[3 * slot:3 * slot + 3] = bytes(trip)
            aa, ok = run(b)
            assert ok == 1, bytes(b)
            assert aa == oracle.translate(bytes(b)), bytes(b)
    # every byte value in every position: canonical iff the byte is one of the ten letters
    base = bytearray(b"ACGTUacgtuAC")
    for pos in range(12):
        for v in range(256):
            b = bytearray(base)
            b[pos] = v
            aa, ok = run(b)
            assert ok == (1 if v in canonical else 0), (pos, v)
            if ok:
                assert aa == oracle.translate(bytes(b))
    # random byte strings
    for _ in range(20000):
        b = bytes(rng.choice(b"ACGTUacgtuNn-@BDHKXxY\x00\xff\x41\x61") for _ in range(12))
        aa, ok = run(b)
        assert ok == (1 if all(c in canonical for c in b) else 0), b
        if ok:
            assert aa == oracle.translate(b), b
