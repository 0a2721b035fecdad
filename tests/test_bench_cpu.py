"""CPU tests of bench.py's reference arm (the driver runs it on the GPU box beside the product's arm): one JSON line
on stdout with the contract's keys, never the product library, rank 0 only under torchrun."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMPED = ("table", "offsets", "data", "counts")


def bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def load_dump(d):
    """A --dump-outputs directory -> (table.npy, {sampled key: count})."""
    import numpy as np
    arr = {n: np.load(os.path.join(d, n + ".npy")) for n in DUMPED}
    assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in DUMPED)
    assert all(a.dtype in (np.float32, np.float64) for a in arr.values())
    assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64 << 20
    raw = arr["data"].astype(np.uint8).tobytes()
    o = arr["offsets"].astype(np.int64)
    keys = [raw[o[i]:o[i + 1]] for i in range(len(arr["counts"]))]
    assert keys == sorted(keys) and len(set(keys)) == len(keys)
    return arr["table"], dict(zip(keys, arr["counts"].astype(int).tolist()))


def expected_dump(bench, table_columns):
    """(table.npy, {sampled key: count}) that --dump-outputs must write for a table given as (offsets, data, counts)."""
    import numpy as np
    (cs, rows, counted), sample = bench.table_sample(np, *table_columns)
    return [rows, counted, cs & 0xFFFFFFFF, cs >> 32], {k: c for _, k, c in sorted(sample)[:bench.DUMP_ROWS]}


def _run(extra_env=None, *args):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--ref-reads", "40000", *args], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout


def test_reference_arm_prints_one_contract_line():
    out = _run()
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "reads/sec" and d["unit"] == "reads/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0
    assert abs(d["value"] - 40000 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["config"]["workload"].startswith("C3") and d["config"]["reads_per_step"] == 40000
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] == (os.cpu_count() or 1)
    assert "NOT parasail" in cb["kind_note"] and cb["sample"] and cb["gcups"] > 0
    # the scalar leg of the same port beside it: same work, one alignment at a time
    assert cb["scalar"]["value"] > 0 and cb["scalar"]["gcups"] > 0


def test_reference_arm_other_configs_and_ranks():
    d = json.loads(_run(None, "--config", "C5"))
    assert d["config"]["workload"].startswith("C5") and d["config"]["adapter_len"] == 40
    # under torchrun only rank 0 runs and prints; the other ranks exit 0 without work
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2").strip() == ""
    d = json.loads(_run({"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"}, "--gpus", "2"))
    assert d["n_gpus"] == 2 and d["impl"] == "reference"


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_reference_arm_dumps_its_last_table(tmp_path):
    """--dump-outputs: the last timed step's table as float arrays, the same whatever the number of steps, and the
    oracle's table for the same reads (40000 reads: fewer rows than the sample holds, so all of them)."""
    import numpy as np
    import oracle
    bench = bench_module()
    _run(None, "--dump-outputs", str(tmp_path / "a"))
    _run(None, "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "b"))
    for n in DUMPED:
        assert np.array_equal(np.load(tmp_path / "a" / (n + ".npy")), np.load(tmp_path / "b" / (n + ".npy")))
    table, rows = load_dump(tmp_path / "a")
    conf = bench.CONFIGS["C3"]
    cfg = oracle.synth_cfg(**conf["synth"])
    p = oracle.make_params(oracle.synth_adapters(cfg), accept_prefix_alignment=conf["thr"], accept_suffix_alignment=conf["thr"])
    text, off, ln = oracle.synth_reads(cfg, 0, 40000)
    want = oracle.process_reads(p, text, off, ln, n_threads=4)[0]
    assert rows == want and list(table[:2]) == [len(want), sum(want.values())]
    assert list(table) == expected_dump(bench, oracle.process_reads(p, text, off, ln, n_threads=4, as_dict=False)[0])[0]


def test_dump_is_independent_of_row_order_and_ranks(tmp_path):
    """The sample is chosen by key hash: a table split over three ranks in another row order dumps the same arrays."""
    import random

    import numpy as np
    bench = bench_module()
    rng = random.Random(5)
    keys = list({bytes(rng.choice(b"ACDEFGHIKLMNPQRSTVWY*") for _ in range(rng.randint(0, 70))) for _ in range(3000)})
    counts = [rng.randint(1, 1000) for _ in keys]

    def columns(idx):
        offs = np.cumsum([0] + [len(keys[i]) for i in idx]).astype(np.uint64)
        return offs, np.frombuffer(b"".join(keys[i] for i in idx), dtype=np.uint8), np.array([counts[i] for i in idx], np.uint64)

    whole = list(range(len(keys)))
    bench.dump_outputs(np, str(tmp_path / "one"), [bench.table_sample(np, *columns(whole), n_rows=500)], n_rows=500)
    rng.shuffle(whole)
    bench.dump_outputs(np, str(tmp_path / "three"), [bench.table_sample(np, *columns(whole[r::3]), n_rows=500) for r in range(3)],
                       n_rows=500)
    for n in DUMPED:
        assert np.array_equal(np.load(tmp_path / "one" / (n + ".npy")), np.load(tmp_path / "three" / (n + ".npy")))
    table, rows = load_dump(tmp_path / "one")
    assert len(rows) == 500 and all(dict(zip(keys, counts))[k] == c for k, c in rows.items())
    assert list(table[:2]) == [len(keys), sum(counts)]


def test_oracle_file_leg(tmp_path):
    """The ingest legs' CPU baseline: the port on a gzipped FASTQ file, phases timed, same table as the plain file call."""
    bench = bench_module()
    import oracle
    cfg = oracle.synth_cfg(seed=5, read_len=150, adapter_len=20, region_len=99, n_variants=500)
    ad = oracle.synth_adapters(cfg)
    leg = bench.oracle_file_leg(oracle, cfg, ad, 0.75, str(tmp_path), 30000, 2)
    assert leg["value"] > 0 and leg["value_if_overlapped"] >= leg["value"] and leg["cores"] == 2 and leg["kind"] == "port"
    assert abs(leg["seconds_inflate_one_zlib_stream"] + leg["seconds_fastq_framing"] + leg["seconds_closures_all_threads_avx2"]
               - leg["seconds"]) < 0.25 * leg["seconds"] + 0.05
    assert os.listdir(tmp_path) == []
    path = str(tmp_path / "same.fq.gz")
    oracle.write_fastq(cfg, 0, 30000, path, bgzf=True, level=1)
    assert leg["table_rows"] == len(oracle.find_variants_file(path, ad, n_threads=2))
