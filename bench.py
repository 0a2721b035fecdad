#!/usr/bin/env python
"""Benchmark of the variant-recovery hot path (BASELINE.json metric: reads/sec, 250-bp synthetic).

    python bench.py --gpus N --steps K --warmup W            # this build, N GPUs (torchrun for N>1)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)
    python bench.py --config C2|C3|C4|C5 ...                 # another BASELINE config (C3 is the headline)
    python bench.py --scaling strong ...                     # the config's reads split over the ranks
    python bench.py --dump-outputs DIR ...                   # also write the last timed step's table as DIR/*.npy

Workload (config.workload): BASELINE config #3 — 100 M synthetic 250-bp merged amplicon reads
per GPU, 20-nt adapters, 30 % of adapters mutated with at least one indel (alignment-heavy),
seed 1003 (SURVEY.md §8(d)); weak scaling: every rank gets its own shard of the same stream.
One step = one pass of the whole hot path (K1 scan -> K2 DP -> K3 translate -> K4 count, then
the table merge over NCCL inside the library when N > 1) over that shard.

Prints ONE JSON line (rank 0).  `value` times the path with reads resident in HBM; `e2e`
times the same reads through the C ABI from pinned HOST buffers (H2D copies and the D2H of
the result table inside the timed region); `ingest` times the user-facing call
`find_variants(path, ..., devices=[0..N-1])` on block-gzip FASTQ files (one process drives all N GPUs).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALU_OPS_PER_CELL = 4    # VIADDMNMX x2 + VIMNMX3 + LOP3 on the INT32 ALU pipe (3 IMAD ride the FMA pipe)
FILTER_ALU_OPS_PER_COL = 11   # k2_filter: 7 LOP3 + PRMT + 2 LEA.HI (score) + VIMNMX per read column

# BASELINE.json configs 2-5 made concrete (SURVEY §8(d)); `reads` = reads per GPU of the resident leg (C4 / C5: the
# per-GPU share at the 8 GPUs the config names).  Scoring is the reference's default 3/-2/5/2 everywhere.
CONFIGS = {
    "C2": dict(workload="C2: 150-bp synthetic reads, 20-nt adapters, 5% adapter errors (exact-match dominated), seed 1002",
               reads=10_000_000, thr=0.75,
               synth=dict(seed=1002, read_len=150, adapter_len=20, region_len=99, n_variants=100000, zipf=1, p_err=0.05,
                          indel=0.5, force_indel=0, frameshift=0.05, noise=0.001, n_rate=1e-4)),
    "C3": dict(workload="C3: 250-bp synthetic merged amplicon reads, 20-nt adapters, 30% adapters mutated (>=1 indel), seed 1003",
               reads=100_000_000, thr=0.75,
               synth=dict(seed=1003, read_len=250, adapter_len=20, region_len=198, n_variants=1000000, zipf=1, p_err=0.30,
                          indel=0.5, force_indel=1, frameshift=0.05, noise=0.001, n_rate=1e-4)),
    "C4": dict(workload="C4: high-diversity library, 250-bp reads drawn uniformly from 10^7 variable regions, 20-nt adapters, "
                        "10% adapter errors, seed 1004 (200 M reads over 8 GPUs = 25 M per GPU)",
               reads=25_000_000, thr=0.75,
               synth=dict(seed=1004, read_len=250, adapter_len=20, region_len=198, n_variants=10000000, zipf=0, p_err=0.10,
                          indel=0.5, force_indel=0, frameshift=0.0, noise=0.0, n_rate=0.0)),
    "C5": dict(workload="C5: 300-bp synthetic reads, 40-nt adapters, 15% adapter errors, thresholds 0.6/0.6, seed 1005 "
                        "(1 B reads over 8 GPUs = 125 M per GPU)",
               reads=125_000_000, thr=0.6,
               synth=dict(seed=1005, read_len=300, adapter_len=40, region_len=210, n_variants=1000000, zipf=1, p_err=0.15,
                          indel=0.5, force_indel=0, frameshift=0.05, noise=0.001, n_rate=1e-4)),
}


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML every
    10 ms from a thread (the timed region of the resident leg is ~0.15 s), `nvidia-smi -lms` if NVML is not importable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None
        self.nv = None
        self.stop_flag = threading.Event()
        self.t = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.nv = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nv
        bits = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))
        while not self.stop_flag.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append(["", sm, self.mx, pw, ""] + ["Active" if rs & b else "Not Active" for _, b in bits])
            except Exception:
                pass
            self.stop_flag.wait(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nv is not None:
            self.stop_flag.set()
            self.t.join(timeout=2)
        elif not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        else:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if str(v).lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvml, 10 ms" if self.nv is not None else "nvidia-smi -lms 50"}


FULL_AFFINITY = None


def bind_to_gpu_cpus(gpu_index):
    """Run this rank on the CPUs NVML names as local to its GPU (the socket its PCIe root hangs off), so that the
    pinned host buffers of the e2e leg are allocated on that NUMA node.  Best effort: containers may forbid it."""
    if os.environ.get("VFB_BENCH_NO_AFFINITY"):
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        global FULL_AFFINITY
        if FULL_AFFINITY is None:
            FULL_AFFINITY = os.sched_getaffinity(0)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = sorted(os.sched_getaffinity(0))
        return "nvml ideal CPUs of GPU %d: %d of %d allowed (%d..%d)" % (gpu_index, len(after), before, after[0], after[-1])
    except Exception as e:
        return "unchanged (%s)" % type(e).__name__


def full_affinity():
    if FULL_AFFINITY is not None:
        try:
            os.sched_setaffinity(0, FULL_AFFINITY)
        except OSError:
            pass


CPU_KIND_NOTE = ("C port of src/lib.rs + parasail's published sg_stats recurrence (oracle/vfind_oracle.c), its alignments run sixteen "
                 "at a time, one 16-bit AVX2 lane per read (oracle/sg_stats_simd.c, bit-identical to the scalar port), exact search "
                 "by the C library's memmem; NOT parasail itself (its AVX2 sg_stats_scan vectorises within one alignment) - "
                 "Rust/parasail cannot be built in this image; `scalar` = the same port one alignment at a time")


def oracle_sample(oracle, adapters, thr, text, off, ln, threads, target_s, simd=True):
    """Time the CPU oracle (all host threads) on a bounded prefix of the workload: (reads, seconds, cells, passes) —
    a prefix that takes about target_s, or, where all of it takes less, several passes over all of it."""
    n_all = len(off)
    probe = min(n_all, 20000 * threads)
    p = oracle.make_params(adapters, accept_prefix_alignment=thr, accept_suffix_alignment=thr)
    t0 = time.perf_counter()
    oracle.process_reads(p, text, off[:probe], ln[:probe], n_threads=threads, simd=simd, as_dict=False)
    dt = time.perf_counter() - t0
    want = probe * target_s / max(dt, 1e-3)
    n = int(min(n_all, max(probe, want)))
    passes = int(max(1, min(64, round(want / n))))
    reads = cells = 0
    t0 = time.perf_counter()
    for _ in range(passes):
        _, _, c = oracle.process_reads(p, text, off[:n], ln[:n], n_threads=threads, simd=simd, as_dict=False)
        reads += n
        cells += c
    dt = time.perf_counter() - t0
    return reads, dt, cells, passes


def cpu_baseline_of(oracle, adapters, thr, text, off, ln, threads, seconds, what):
    """The cpu_baseline object: the SIMD leg of the port (the value) with the scalar leg beside it."""
    cn, cdt, ccells, passes = oracle_sample(oracle, adapters, thr, text, off, ln, threads, seconds, simd=True)
    sn, sdt, scells, sp = oracle_sample(oracle, adapters, thr, text, off, ln, threads, max(2.0, seconds / 4), simd=False)
    return {"value": cn / cdt, "unit": "reads/s", "cores": threads, "kind": "port", "kind_note": CPU_KIND_NOTE,
            "simd": "avx2, 16 alignments per vector" if oracle.simd_available() else "unavailable on this host: scalar",
            "sample": "first %d reads of %s, %d pass(es), %.1f s" % (cn // passes, what, passes, cdt),
            "gcups": ccells / cdt / 1e9,
            "scalar": {"value": sn / sdt, "unit": "reads/s", "gcups": scells / sdt / 1e9,
                       "sample": "first %d reads, %d pass(es), %.1f s" % (sn // sp, sp, sdt)}}


def oracle_file_leg(oracle, cfg, adapters, thr, tmp, n_reads, threads):
    """The CPU port on a gzipped FASTQ FILE, whole call (the ingest legs' baseline): a block-gzip file of the first n_reads
    reads of the stream, inflated by ONE zlib stream (the reference's MultiGzDecoder runs on one reader thread), framed,
    then the closures on every host thread with the AVX2 leg.  The port runs the three phases one after the other; the
    reference overlaps its reader thread with its workers, so `value_if_overlapped` (reads / the longer of the two) is
    the number to hold the GPU path against."""
    path = os.path.join(tmp, "oracle_leg.fq.gz")
    tb, zb = oracle.write_fastq(cfg, 0, n_reads, path, bgzf=True, level=1)
    try:
        t0 = time.perf_counter()
        rows, n, ph = oracle.find_variants_file_timed(path, adapters, n_threads=threads, simd=True,
                                                      accept_prefix_alignment=thr, accept_suffix_alignment=thr)
        dt = time.perf_counter() - t0
    finally:
        os.remove(path)
    reader = ph[0] + ph[1]
    return {"value": n / dt, "unit": "reads/s", "value_if_overlapped": n / max(reader, ph[2], 1e-9), "cores": threads, "kind": "port",
            "input": "block-gzip FASTQ, first %d reads of the stream, %.0f MB text, %.0f MB compressed" % (n, tb / 1e6, zb / 1e6),
            "seconds": dt, "seconds_inflate_one_zlib_stream": ph[0], "seconds_fastq_framing": ph[1],
            "seconds_closures_all_threads_avx2": ph[2], "table_rows": rows,
            "note": "the reference's reader (flate2 MultiGzDecoder + seq_io) is one thread too: from a .gz file it is bound by that "
                    "thread whatever the aligner costs"}


def run_reference(args):
    """--impl reference: the reference's CPU path (the oracle port — the Rust/parasail reference cannot be built in
    this image), all host threads, a bounded sample of the workload per step.  Inputs come from the oracle side's own
    generator (oracle/synth_host.c): this arm never loads libvfind_b200.so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    oracle.build()
    conf = dict(CONFIGS[args.config])
    if args.thr > 0:
        conf["thr"] = args.thr
        conf["workload"] += " [thresholds overridden: %g]" % args.thr
    cfg = oracle.synth_cfg(**conf["synth"])
    adapters = oracle.synth_adapters(cfg)
    threads = os.cpu_count() or 1
    n = args.ref_reads
    text, off, ln = oracle.synth_reads(cfg, 0, n, threads)
    p = oracle.make_params(adapters, accept_prefix_alignment=conf["thr"], accept_suffix_alignment=conf["thr"])
    times = []
    cells = 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        table, _, cells = oracle.process_reads(p, text, off, ln, n_threads=threads, simd=True, as_dict=False)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        import numpy as np
        dump_outputs(np, args.dump_outputs, [table_sample(np, *table)])
    total = sum(times)
    value = n * len(times) / total
    # the same port one alignment at a time, beside it (a short sample, not part of the timed steps)
    s_reads, s_dt, s_cells, s_passes = oracle_sample(oracle, adapters, conf["thr"], text, off, ln, threads, 3.0, simd=False)
    assert "vfind_b200" not in sys.modules, "the reference arm must not load the product"
    line = {
        "impl": "reference", "metric": "reads/sec", "value": value, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int32",
        "data": "synthetic",
        "config": {"workload": conf["workload"], "reads_per_step": n, "read_len": cfg.read_len,
                   "adapter_len": cfg.adapter_len, "thresholds": [conf["thr"], conf["thr"]],
                   "note": "CPU oracle port; bounded sample of the workload; inputs from oracle/synth_host.c"},
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": threads, "kind": "port", "kind_note": CPU_KIND_NOTE,
                         "simd": "avx2, 16 alignments per vector" if oracle.simd_available() else "unavailable on this host: scalar",
                         "sample": "%d reads of the %s stream per step" % (n, args.config),
                         "gcups": cells / (total / len(times)) / 1e9,
                         "scalar": {"value": s_reads / s_dt, "unit": "reads/s", "gcups": s_cells / s_dt / 1e9,
                                    "sample": "first %d reads, %d pass(es), %.1f s, outside the timed steps" % (s_reads // s_passes, s_passes, s_dt)}},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else libraries print on fd 1 (NCCL's version banner,
    for one) was sent to stderr by main()."""
    os.write(REAL_STDOUT, (json.dumps(line) + "\n").encode())


REAL_STDOUT = 1


def key_hashes(np, offsets, data, block_rows=1 << 18):
    """uint64 mix(key bytes, length) of every row of a (sequence, count) table, a block of rows at a time so that a table
    of millions of keys needs no more than a few hundred MB of temporaries."""
    rows = len(offsets) - 1
    out = np.zeros(max(rows, 0), dtype=np.uint64)
    for r0 in range(0, rows, block_rows):
        r1 = min(rows, r0 + block_rows)
        offs = offsets[r0:r1 + 1].astype(np.int64)
        d = data[offs[0]:offs[-1]]
        offs = offs - offs[0]
        lens = (offs[1:] - offs[:-1]).astype(np.int64)
        pos = np.arange(len(d), dtype=np.int64) - np.repeat(offs[:-1], lens)
        w = (pos.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0xD1342543DE82EF95)) | np.uint64(1)
        with np.errstate(over="ignore"):
            terms = (d.astype(np.uint64) + np.uint64(1)) * w
            nz = lens > 0
            rowsum = np.zeros(r1 - r0, dtype=np.uint64)
            if nz.any():
                rowsum[nz] = np.add.reduceat(terms, offs[:-1][nz])
            mixed = (rowsum ^ lens.astype(np.uint64)) * np.uint64(0xBF58476D1CE4E5B9)
            mixed ^= mixed >> np.uint64(29)
        out[r0:r1] = mixed
    return out


def table_checksum(np, offsets, data, counts, hashes=None):
    """Order-independent 64-bit checksum of a (sequence, count) table: sum over rows of mix(key bytes, length) * (2 count + 1)."""
    rows = len(counts)
    if rows == 0:
        return 0, 0, 0
    hashes = key_hashes(np, offsets, data) if hashes is None else hashes
    with np.errstate(over="ignore"):
        total = (hashes * (counts.astype(np.uint64) * np.uint64(2) + np.uint64(1))).sum(dtype=np.uint64)
    return int(total), int(rows), int(counts.sum())


DUMP_ROWS = 1 << 15         # rows of the table --dump-outputs writes: keys of <= 300 bytes as float32 stay under 40 MB
DUMP_SEED = 0x5EED5A3B1E0F


def table_sample(np, offsets, data, counts, n_rows=DUMP_ROWS):
    """What --dump-outputs keeps of a (sequence, count) table: its checksum triple and [(rank hash, key, count)] of the
    n_rows rows of smallest seeded key hash.  Which rows those are depends on the keys alone, not on the table's row order
    or on how its keys are split over ranks, so two builds are compared row for row."""
    k = key_hashes(np, offsets, data)
    with np.errstate(over="ignore"):
        h = (k ^ np.uint64(DUMP_SEED)) * np.uint64(0x94D049BB133111EB)
        h ^= h >> np.uint64(31)
    sel = np.arange(len(h))
    if len(h) > n_rows:
        sel = np.nonzero(h <= np.partition(h, n_rows - 1)[n_rows - 1])[0]
    rows = [(int(h[i]), data[int(offsets[i]):int(offsets[i + 1])].tobytes(), int(counts[i])) for i in sel]
    return table_checksum(np, offsets, data, counts, k), rows


def dump_outputs(np, out_dir, parts, n_rows=DUMP_ROWS):
    """Writes the table the timed path computed, from the table_sample() of every rank's share of it:
    table.npy    float64 [rows, counted reads, checksum bits 0-31, checksum bits 32-63] of the whole table;
    offsets.npy  float64 [n+1], data.npy float32 [key bytes], counts.npy float64 [n]: the sampled rows sorted by key,
                 in the layout of Context.finish_arrays()."""
    checksum = sum(p[0][0] for p in parts) % (1 << 64)
    rows = sorted((r for p in parts for r in p[1]))[:n_rows]       # the global smallest hashes; ties are 1 in 2^64
    rows.sort(key=lambda r: r[1])
    lens = [len(r[1]) for r in rows]
    arrays = {
        "table": np.array([sum(p[0][1] for p in parts), sum(p[0][2] for p in parts), checksum & 0xFFFFFFFF, checksum >> 32],
                          dtype=np.float64),
        "offsets": np.concatenate([[0], np.cumsum(lens)]).astype(np.float64),
        "data": np.frombuffer(b"".join(r[1] for r in rows), dtype=np.uint8).astype(np.float32),
        "counts": np.array([r[2] for r in rows], dtype=np.float64),
    }
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def traffic_record(kernel_file_of):
    """DRAM bytes per launch from the committed ncu capture (profiles/r02_ncu_traffic.json), valid only while the
    kernel's source file is the one the capture was taken from (sha1 recorded at capture time)."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
    except (OSError, ValueError):
        return {}, "no capture committed"
    out = {}
    for k, v in rec.get("kernels", {}).items():
        path = os.path.join(ROOT, "vfind_b200", "csrc", v.get("file", kernel_file_of.get(k, "")))
        try:
            sha = hashlib.sha1(open(path, "rb").read()).hexdigest()
        except OSError:
            sha = None
        out[k] = v["dram_bytes"] if sha and sha == v.get("sha1") else None
    return out, "ncu --set full, %s, commit %s, %d reads per launch; null = the kernel file changed since" % (
        rec.get("when", "?"), rec.get("commit", "?"), rec.get("reads_per_launch", 0))


def main():
    global REAL_STDOUT
    sys.stdout.flush()
    REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C3", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --reads per GPU; strong: --reads in total, split over the ranks")
    ap.add_argument("--thr", type=float, default=0.0, help="override the config's accept thresholds (both adapters)")
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU per step (strong: in total); 0 = the config's")
    ap.add_argument("--chunk-reads", type=int, default=12_500_000)
    ap.add_argument("--e2e-reads", type=int, default=-1, help="reads per e2e step (-1 = same as --reads)")
    ap.add_argument("--ref-reads", type=int, default=4_000_000, help="reads per step of --impl reference")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--ingest-reads", type=int, default=50_000_000,
                    help="reads in the block-gzip FASTQ file of the ingest leg (0 = skip)")
    ap.add_argument("--ingest-block", type=int, default=10_000_000,
                    help="distinct reads generated for the ingest file; the file repeats this block up to --ingest-reads")
    ap.add_argument("--ingest-c5-reads", type=int, default=30_000_000, help="reads in the C5-shaped ingest file (0 = skip)")
    ap.add_argument("--table-hint", type=int, default=40_000_000, help="expected distinct variants per GPU (table capacity hint)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the table of the last step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from vfind_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = bind_to_gpu_cpus(local)          # before any pinned allocation: first touch decides the NUMA node
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        idle_group = dist.new_group(backend="gloo")     # the ranks that sit out the ingest leg wait on sockets, not on a spinning kernel
        # the table merge runs inside the library over its own NCCL communicator; torch.distributed only carries
        # the 128-byte id (and the timing reductions of this script)
        ids = [api.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = api.nccl_comm_init(ids[0], world, rank, local)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node = --gpus"

    conf = dict(CONFIGS[args.config])
    if args.thr > 0:
        conf["thr"] = args.thr
        conf["workload"] += " [thresholds overridden: %g]" % args.thr
    cfg = api.synth_cfg(**conf["synth"])
    thr = conf["thr"]
    adapters = api.synth_adapters(cfg)
    R_cfg = args.reads if args.reads > 0 else conf["reads"]
    R = R_cfg if args.scaling == "weak" else (R_cfg + world - 1) // world       # reads of this rank per step
    L = cfg.read_len
    ctx_kw = dict(accept_prefix_alignment=thr, accept_suffix_alignment=thr)
    # ---- synthetic shard of this rank, resident in HBM, in <= 4 GiB chunks
    chunks = []
    first = rank * R
    done = 0
    while done < R:
        n = min(args.chunk_reads, R - done)
        t = torch.empty(n * L, dtype=torch.uint8, device=dev)
        s = torch.empty(n * 2, dtype=torch.int32, device=dev)
        api.synth_device(cfg, first + done, n, t.data_ptr(), s.data_ptr(), local)
        chunks.append((t, s, n))
        done += n
    torch.cuda.synchronize()

    stream = torch.cuda.Stream(device=dev)
    ctx = api.Context(adapters, device=local, table_capacity_hint=min(R, args.table_hint), batch_reads=args.chunk_reads, **ctx_kw)
    ctx.set_compute_stream(stream.cuda_stream)

    merge_events = []

    def step_device():
        ctx.table_clear()
        for t, s, n in chunks:
            ctx.submit_device(t.data_ptr(), t.numel(), s.data_ptr(), n)
        if world > 1:
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ctx.fence()
            m0.record(stream)
            ctx.merge_nccl(comm, rank, world)
            m1.record(stream)
            merge_events.append((m0, m1))

    def barrier():
        stream.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_device()
        barrier()
        merge_check = None
        if world > 1:
            # untimed check of the merge: the same 2 M reads once on one GPU (rank 0) and once split over the ranks and
            # merged; the merged partitions must add up to exactly the one-GPU table (order-independent checksum over
            # keys and counts, rows, counted reads)
            n_chk = min(2_000_000, R * world)
            per = (n_chk + world - 1) // world
            lo = min(rank * per, n_chk)
            m = min(per, n_chk - lo)
            ctx.table_clear()
            if m:
                ht, hs = api.synth_host(cfg, lo, m)
                ctx.submit_host(ht, hs)
            ctx.merge_nccl(comm, rank, world)
            cs = table_checksum(np, *ctx.finish_arrays(copy=False))
            parts = [None] * world
            dist.all_gather_object(parts, cs)
            if rank == 0:
                ctx.table_clear()
                ht, hs = api.synth_host(cfg, 0, n_chk)
                ctx.submit_host(ht, hs)
                one = table_checksum(np, *ctx.finish_arrays(copy=False))
                merged = (sum(p[0] for p in parts) % (1 << 64), sum(p[1] for p in parts), sum(p[2] for p in parts))
                merge_check = {"reads": n_chk, "one_gpu": {"checksum": one[0], "rows": one[1], "counted": one[2]},
                               "merged": {"checksum": merged[0], "rows": merged[1], "counted": merged[2]},
                               "rows_per_rank": [p[1] for p in parts], "ok": tuple(one) == merged}
            barrier()
        ctx.reset()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        merge_events.clear()
        e0.record(stream)
        for _ in range(args.steps):
            step_device()
        ctx.fence()                      # the library's lane streams join the compute stream before the end event
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        merge_ms = sum(a.elapsed_time(b) for a, b in merge_events) / max(1, len(merge_events)) if merge_events else 0.0
        clocks = sampler.stop() if rank == 0 else None
        st_timed = ctx.stats()
        if args.dump_outputs:
            # the table of the last timed step; after the merge each rank holds the keys it owns
            part = table_sample(np, *ctx.finish_arrays(copy=False))
            parts = [part] if world == 1 else [None] * world
            if world > 1:
                dist.all_gather_object(parts, part)
            if rank == 0:
                dump_outputs(np, args.dump_outputs, parts)
        # per-kernel times for the rooflines: the same steps once more with the batches back to back on ONE stream
        # (in the timed region above consecutive batches overlap on two lanes, so a kernel's duration there includes
        # whatever shared the SMs with it)
        ctx.set_lanes(1)
        ctx.reset()
        ctx.set_profiling(True)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(stream)
        for _ in range(args.steps):
            step_device()
        p1.record(stream)
        barrier()
        serial_ms = p0.elapsed_time(p1) / args.steps
        st = ctx.stats()
        ctx.set_profiling(False)
        ctx.set_lanes(2)
        tms = torch.tensor([ms, merge_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms_max, merge_ms = float(tms[0].item()), float(tms[1].item())
        value = world * R * args.steps / (ms_max * 1e-3)

        # ---- e2e: the same reads from pinned host memory through vfb_submit_host + vfb_finish
        e2e = None
        if not args.no_e2e:
            er = R if args.e2e_reads < 0 else min(args.e2e_reads, R)
            host = []
            got = 0
            for t, s, n in chunks:
                if got >= er:
                    break
                m = min(n, er - got)
                ht = torch.empty(m * L, dtype=torch.uint8, pin_memory=True)
                hs = torch.empty(m * 2, dtype=torch.int32, pin_memory=True)
                ht.copy_(t[:m * L]); hs.copy_(s[:m * 2])
                host.append((ht, hs, m))
                got += m
            torch.cuda.synchronize()
            rows = 0

            def step_e2e():
                nonlocal rows
                ctx.table_clear()
                for ht, hs, m in host:
                    ctx.submit_host_ptr(ht.data_ptr(), ht.numel(), hs.data_ptr(), m)
                if world > 1:
                    ctx.merge_nccl(comm, rank, world)
                offsets, data, counts = ctx.finish_arrays(copy=False)
                rows = len(counts)
                return offsets.nbytes + data.nbytes + counts.nbytes

            step_e2e()
            barrier()
            # what bounds it, measured: the link alone (one pinned chunk copied by itself, best of 3) and the host's
            # own memory (one thread copying the same pinned chunk to another pinned buffer)
            link_gbs = host_gbs = 0.0
            if host:
                ht0 = host[0][0]
                scratch = torch.empty(ht0.numel(), dtype=torch.uint8, device=dev)
                for _ in range(3):
                    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    c0.record(stream)
                    scratch.copy_(ht0, non_blocking=True)
                    c1.record(stream)
                    stream.synchronize()
                    link_gbs = max(link_gbs, ht0.numel() / (c0.elapsed_time(c1) * 1e-3) / 1e9)
                del scratch
                nb = min(ht0.numel(), 1 << 30)
                dst = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
                for _ in range(2):
                    t0 = time.perf_counter()
                    dst.copy_(ht0[:nb])
                    host_gbs = max(host_gbs, nb / (time.perf_counter() - t0) / 1e9)
                del dst
            barrier()
            d2h = 0
            link0 = ctx.stats()["h2d_bytes"]
            t0 = time.perf_counter()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            esteps = args.steps
            for _ in range(esteps):
                d2h = step_e2e()
            f1.record(stream)
            barrier()
            wall = time.perf_counter() - t0
            link_bytes = (ctx.stats()["h2d_bytes"] - link0) / esteps
            ems = torch.tensor([max(f0.elapsed_time(f1), wall * 1e3)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(ems, op=dist.ReduceOp.MAX)
            step_ms = float(ems.item()) / esteps
            h2d_step = int(sum(h[0].numel() + h[1].numel() * 4 for h in host))
            per_gpu_gbs = h2d_step / (step_ms * 1e-3) / 1e9
            kernels_ms = ms_max / args.steps * (got / R)
            frac = per_gpu_gbs / link_gbs if link_gbs else 0.0
            if frac >= 0.85:
                bound = "PCIe link: %.1f GB/s per GPU inside the step vs %.1f GB/s for one chunk copied alone" % (per_gpu_gbs, link_gbs)
            elif world > 1:
                bound = ("host memory / root complex shared by %d GPUs: %.1f GB/s per GPU inside the step (%.1f GB/s in total) vs %.1f GB/s "
                         "for one chunk copied alone on one GPU" % (world, per_gpu_gbs, per_gpu_gbs * world, link_gbs))
            else:
                bound = ("host side of the copy: %.1f GB/s inside the step vs %.1f GB/s for one chunk copied alone (a host thread "
                         "copies pinned memory at %.1f GB/s here); the kernels need %.0f of the step's %.0f ms"
                         % (per_gpu_gbs, link_gbs, host_gbs, kernels_ms, step_ms))
            e2e = {"value": world * got * esteps / (float(ems.item()) * 1e-3), "unit": "reads/s",
                   "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": int(d2h), "reads_per_step": got, "steps": esteps,
                   "table_rows": rows, "ms_per_step": step_ms,
                   "h2d_gbs_achieved": world * per_gpu_gbs, "h2d_gbs_per_gpu": per_gpu_gbs,
                   "h2d_gbs_link_alone": link_gbs, "host_memcpy_gbs_one_thread": host_gbs,
                   "h2d_bytes_on_link_per_step": int(link_bytes), "kernels_ms_per_step": kernels_ms,
                   "bound": bound, "bound_how": "computed from the three rates measured in this run"}
            del host

    # ---- every rank lets go of its device memory: the ingest leg (rank 0) drives ALL GPUs from one process
    st_reads = st["reads"]
    try:
        del t, s
    except NameError:
        pass
    chunks.clear()
    ctx.close()
    torch.cuda.empty_cache()
    api.load_library().vfb_device_pool_trim()
    if world > 1:
        barrier()

    if rank != 0:
        if world > 1:
            api.nccl_comm_destroy(comm)
            dist.barrier(group=idle_group)              # rank 0's ingest leg
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (K2 DP, INT32-ALU bound) and of the HBM-bound scan
    alu_gops, dual_gops = api.measure_int_peak(local)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    traffic, traffic_how = traffic_record({"k2_dp_window": "kernels_dpw.cu", "k2_filter": "kernels_dpw.cu", "k1_scan": "kernels_scan.cu"})
    if args.config != "C3" or min(args.chunk_reads, R) != 12_500_000:
        traffic = {}                    # captured on C3 at 12.5 M reads per launch: not comparable otherwise
    dp_s = st["ms_dp"] * 1e-3
    gcups = st["dp_cells"] / dp_s / 1e9 if dp_s > 0 else 0.0      # effective: full A x L matrices / DP stage time
    windowed = st["dp_kernel_kind"] == 3
    if windowed:
        # the DP stage = k2_filter (Myers bit-vector, every column of every aligned read) + k2_dp_window
        # (packed Gotoh cells on the flagged windows only) + k2_resolve.  Roofline of the window kernel:
        # cells it actually evaluated x 4 ALU-pipe ops, against the measured ALU-pipe peak.
        win_s = st["ms_dp_window"] * 1e-3
        kernel_gcups = st["dp_cells_computed"] / win_s / 1e9 if win_s > 0 else 0.0
        dp_kernel, dp_ms = "k2_dp_window", st["ms_dp_window"]
    else:
        kernel_gcups, dp_kernel, dp_ms = gcups, "k2_dp_packed", st["ms_dp"]
    dp_achieved = kernel_gcups * ALU_OPS_PER_CELL     # G lane-ops/s on the ALU pipe
    scan_bytes = st_reads * (L + 12)                  # SURVEY §8(d): N*(L+12)
    scan_gbs = scan_bytes / (st["ms_scan"] * 1e-3) / 1e9 if st["ms_scan"] > 0 else 0.0
    # every step starts from a cleared table (counters included): `counted` / `unique` / `fused_hits` are one step's
    key_bytes = st["counted"] * args.steps * (cfg.region_len + cfg.region_len // 3 + 8)
    roofline = {"bound": "int32", "kernel": dp_kernel, "achieved": dp_achieved, "peak": alu_gops,
                "unit": "Gop/s", "frac": dp_achieved / alu_gops if alu_gops else None,
                "traffic": traffic.get(dp_kernel), "traffic_unit": "DRAM bytes per launch", "traffic_how": traffic_how,
                "gcups": kernel_gcups, "alu_ops_per_cell": ALU_OPS_PER_CELL,
                "peak_source": "vfb_measure_int_peak (VIADDMNMX stream, measured in this run); ALU+FMA dual-issue peak %.0f Gop/s" % dual_gops,
                "share_of_step": dp_ms / st["ms_total"] if st["ms_total"] else None}
    roofline_filter = None
    if windowed and st["ms_dp_filter"] > 0:
        # Myers column: 7 LOP3 + 1 PRMT + 3 score/min ops on the ALU pipe (3 IMAD adds/shifts on the FMA pipe, 1 LDS)
        cols = st["dp_cells"] / cfg.adapter_len       # one column per read base of every aligned read
        f_ach = cols * FILTER_ALU_OPS_PER_COL / (st["ms_dp_filter"] * 1e-3) / 1e9
        roofline_filter = {"bound": "int32", "kernel": "k2_filter", "achieved": f_ach, "peak": alu_gops, "unit": "Gop/s",
                           "frac": f_ach / alu_gops if alu_gops else None, "traffic": traffic.get("k2_filter"),
                           "columns_per_s": cols / (st["ms_dp_filter"] * 1e-3), "alu_ops_per_column": FILTER_ALU_OPS_PER_COL,
                           "share_of_step": st["ms_dp_filter"] / st["ms_total"] if st["ms_total"] else None}
    roofline_hbm = {"bound": "hbm", "kernel": "k1_scan", "achieved": scan_gbs, "peak": hbm_peak, "unit": "GB/s",
                    "frac": scan_gbs / hbm_peak, "traffic": traffic.get("k1_scan"),
                    "algorithmic_bytes_per_launch": min(args.chunk_reads, R) * (L + 12), "peak_source": hbm_src,
                    "share_of_step": st["ms_scan"] / st["ms_total"] if st["ms_total"] else None}
    stages = {k: st[k] / args.steps for k in ("ms_scan", "ms_worklist", "ms_dp", "ms_dp_filter", "ms_dp_window",
                                              "ms_translate", "ms_count", "ms_total")}
    stages["translate_gbs"] = key_bytes / (st["ms_translate"] * 1e-3) / 1e9 if st["ms_translate"] > 0 else 0.0
    count_bytes = (st["counted"] * (cfg.region_len // 3 + 24) + st["unique"] * (cfg.region_len // 3 + 8)) * args.steps
    stages["count_gbs"] = count_bytes / (st["ms_count"] * 1e-3) / 1e9 if st["ms_count"] > 0 else 0.0

    import oracle
    oracle.build()
    cpu = None
    if world == 1 and not args.no_cpu:
        full_affinity()                                 # the CPU baseline gets every host core
        threads = os.cpu_count() or 1
        m = min(R, 4_000_000)
        text, off, ln = oracle.synth_reads(cfg, 0, m, threads)
        cpu = cpu_baseline_of(oracle, adapters, thr, text, off, ln, threads, args.cpu_seconds, "the same %s stream" % args.config)
        del text, off, ln

    # ---- ingest legs: the user-facing call, vfind.find_variants(path, adapters, devices=[0..N-1]) — ONE process drives all
    # N GPUs — on block-gzip FASTQ files: file read, H2D of the compressed members, GPU inflate, GPU FASTQ parse, K1..K4,
    # table merge over peer copies, table hand-off; whole call.  Files: the config's stream (a block of distinct reads
    # repeated up to the file size, SURVEY §8(d)), and a C5-shaped one (300 bp, 40-nt adapters, 0.6/0.6).
    ingest = None
    if args.ingest_reads > 0:
        full_affinity()
        ingest = {}
        try:
            import tempfile
            from vfind_b200 import find_variants
            tmp = tempfile.mkdtemp(prefix="vfb_bench_")
            devs = list(range(world))

            def make_file(name, conf_k, n_reads, block):
                c = oracle.synth_cfg(**conf_k["synth"])
                path = os.path.join(tmp, name)
                t0 = time.perf_counter()
                block = min(block, n_reads)
                reps = max(1, n_reads // block)
                one = path + ".block"
                tb, zb = oracle.write_fastq(c, 0, block, one, bgzf=True, level=1, append=True)    # no end-of-file member yet
                with open(path, "wb") as out:
                    for _ in range(reps):
                        with open(one, "rb") as src:
                            while True:
                                buf = src.read(64 << 20)
                                if not buf:
                                    break
                                out.write(buf)
                os.remove(one)
                oracle.write_fastq(c, 0, 0, path, bgzf=True, level=1, append=True)               # the empty end-of-file member
                return path, block * reps, tb * reps, os.path.getsize(path), reps, time.perf_counter() - t0, c

            def time_calls(path, ads, kw, n_reads, reps=3):
                times, rows, total = [], 0, 0
                for rep in range(reps + 1):
                    t0 = time.perf_counter()
                    out = find_variants(path, ads, show_progress=False, devices=devs, **kw)
                    times.append(time.perf_counter() - t0)
                    rows = out.num_rows if hasattr(out, "num_rows") else len(out)
                    if rep == 0:
                        col = out.column("count") if hasattr(out, "column") else out["count"]
                        total = int(np.asarray(col.to_numpy() if hasattr(col, "to_numpy") else col).sum())
                    del out
                return min(times[1:]), times[0], rows, total

            legs = [("stream", conf, args.ingest_reads, args.ingest_block)]
            if args.ingest_c5_reads > 0 and args.config != "C5":
                legs.append(("c5_shape", CONFIGS["C5"], args.ingest_c5_reads, args.ingest_block))
            for name, conf_k, n_reads, block in legs:
                path, n_file, tb, zb, reps, gen_s, c = make_file(name + ".fq.gz", conf_k, n_reads, block)
                ads = tuple(a.decode() for a in oracle.synth_adapters(c))
                kw = dict(accept_prefix_alignment=conf_k["thr"], accept_suffix_alignment=conf_k["thr"])
                best, first_call, rows, counted = time_calls(path, ads, kw, n_file)
                leg = {"value": n_file / best, "unit": "reads/s", "call": "vfind.find_variants(path, adapters, devices=%r)" % devs,
                       "n_gpus": world, "reads_per_min": 60.0 * n_file / best,
                       "input": "block-gzip (BGZF, zlib level 1) FASTQ, %d reads (%d x a block of %d distinct reads), %.1f GB text, %.2f GB compressed, "
                                "generated in %.0f s" % (n_file, reps, n_file // reps, tb / 1e9, zb / 1e9, gen_s),
                       "seconds_best_of_3": best, "seconds_first_call": first_call, "table_rows": rows, "counted_reads": counted,
                       "text_gbs": tb / best / 1e9, "compressed_gbs": zb / best / 1e9}
                if name == "stream":
                    ingest.update(leg)
                else:
                    ingest[name] = leg
                os.remove(path)
            if world == 1 and not args.no_cpu:
                try:
                    full_affinity()
                    ingest["cpu_baseline"] = oracle_file_leg(oracle, cfg, adapters, thr, tmp, min(args.ingest_reads, 2_000_000),
                                                             os.cpu_count() or 1)
                except Exception as e:
                    ingest["cpu_baseline"] = {"error": repr(e)}
            if world == 1:
                # the same call on ONE plain gzip stream (what `gzip` / pigz / fastp write): decoded on the device
                # (block-start search, marker decode, resolve: kernels_inflate.cu k_gz_*), and for comparison by the
                # parallel host gunzip (pgunzip.cu) on the ingest threads (VFB_GPU_GUNZIP=0)
                n_gz = min(args.ingest_reads, 8_000_000)
                txt = os.path.join(tmp, "plain.fq")
                gz = txt + ".gz"
                tb2, _ = oracle.write_fastq(cfg, 0, n_gz, txt, bgzf=False)
                subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "single_stream_gzip.py"), txt, gz, "1"])
                os.remove(txt)
                ads = tuple(a.decode() for a in adapters)
                legs = {}
                for mode in ("1", "0"):
                    os.environ["VFB_GPU_GUNZIP"] = mode
                    times = []
                    for rep in range(3):
                        t0 = time.perf_counter()
                        find_variants(gz, ads, show_progress=False, device=0, accept_prefix_alignment=thr, accept_suffix_alignment=thr)
                        times.append(time.perf_counter() - t0)
                    legs[mode] = min(times)
                    legs[mode + "_all"] = [round(x, 4) for x in times]
                os.environ.pop("VFB_GPU_GUNZIP", None)
                ingest["plain_gzip"] = {"value": n_gz / legs["1"], "unit": "reads/s",
                                        "input": "ONE gzip member holding one deflate stream (zlib level 1, written in parallel slices "
                                                 "that end with a sync flush, as pigz does), %d reads, %.0f MB text, %.0f MB compressed"
                                                 % (n_gz, tb2 / 1e6, os.path.getsize(gz) / 1e6),
                                        "decoder": "device (k_gz_search / k_gz_decode / k_gz_chain / k_gz_resolve)",
                                        "seconds_best_of_3": legs["1"], "seconds_all": legs["1_all"],
                                        "host_threads_value": n_gz / legs["0"], "host_threads": min(os.cpu_count() or 1, 32),
                                        "host_threads_seconds_best_of_3": legs["0"], "host_threads_seconds_all": legs["0_all"]}
                os.remove(gz)
            os.rmdir(tmp)
        except Exception as e:          # the ingest leg never fails the bench line
            ingest["error"] = repr(e)

    line = {
        "metric": "reads/sec", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": conf["workload"], "config": args.config, "reads_per_gpu": R, "reads_total_per_step": R * world,
                   "read_len": L, "adapter_len": cfg.adapter_len,
                   "region_len": cfg.region_len, "library": cfg.n_variants, "thresholds": [thr, thr],
                   "scoring": [3, -2, 5, 2], "l2": "inputs (%.1f GB per GPU) are larger than L2" % (R * L / 1e9),
                   "parallelism": "reads sharded over %d GPU(s), keep-own-keys table merge over NCCL send/recv inside the library" % world,
                   "cpu_affinity": affinity},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(st_timed["kernel_launches"]),
        "lanes": {"timed_region": "consecutive batches overlap on 2 lane streams (only the table insert is serialised)",
                  "ms_per_step_one_lane": serial_ms,
                  "stages_and_rooflines": "from %d extra steps with the batches back to back on one stream" % args.steps},
        "roofline": roofline, "roofline_filter": roofline_filter, "roofline_hbm": roofline_hbm,
        "stages_ms_per_step": stages,
        "dp": {"effective_gcups": gcups, "mode": "windowed (filter + windows)" if windowed else "full matrices",
               "cells_per_step": st["dp_cells"] // args.steps,
               "cells_computed_per_step": st["dp_cells_computed"] // args.steps,
               "windows_per_step": st["dp_windows"] // args.steps,
               "alignments_per_step": (st["dp_prefix"] + st["dp_suffix"]) // args.steps},
        "merge_ms_per_step": merge_ms, "table": {"unique": st["unique"], "counted_per_step": st["counted"],
                                                        "counted_by_the_key_kernel_per_step": st.get("fused_hits", 0),
                                                        "fused_key_count": bool(st.get("fused_batches", 0)), "merge_check": merge_check},
        "cpu_baseline": cpu, "ingest": ingest,
    }
    emit(line)
    if world > 1:
        api.nccl_comm_destroy(comm)
        dist.barrier(group=idle_group)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
