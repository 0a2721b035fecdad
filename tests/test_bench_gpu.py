"""bench.py's product arm at a small size: the line reports the steps it was asked for, and --dump-outputs writes the
table of the last timed step, which is the CPU oracle's table for the same reads."""
import json
import os
import subprocess
import sys

import pytest

import oracle
from test_bench_cpu import ROOT, bench_module, expected_dump, load_dump

pytestmark = pytest.mark.gpu


def test_dump_outputs_match_the_oracle(tmp_path):
    n = 300_000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--reads", str(n), "--chunk-reads", "100000", "--table-hint", "1000000", "--no-cpu",
                        "--ingest-reads", "0", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout)
    assert d["steps"] == 2 and d["e2e"]["steps"] == 2 and d["config"]["reads_per_gpu"] == n
    table, rows = load_dump(tmp_path / "out")
    bench = bench_module()
    conf = bench.CONFIGS["C3"]
    cfg = oracle.synth_cfg(**conf["synth"])
    p = oracle.make_params(oracle.synth_adapters(cfg), accept_prefix_alignment=conf["thr"], accept_suffix_alignment=conf["thr"])
    text, off, ln = oracle.synth_reads(cfg, 0, n)
    want_table, want_rows = expected_dump(bench, oracle.process_reads(p, text, off, ln, n_threads=os.cpu_count() or 1,
                                                                      as_dict=False)[0])
    assert list(table) == want_table and table[1] == d["table"]["counted_per_step"]
    assert len(rows) == min(bench.DUMP_ROWS, want_table[0]) and rows == want_rows
