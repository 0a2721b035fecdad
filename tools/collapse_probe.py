"""Cost of collapse_ratio on C3-shaped count tables.

    python tools/collapse_probe.py [--reads 10000000,100000000] [--ratio 2] [--sample 5000] [--out DIR]

For each read count and skip_translation off / on, C3 reads (250-bp synthetic amplicons, 20-nt adapters, 198-nt region,
1 M library members, 0.1 % per-base region noise, 1e-4 N calls) are generated on the device and counted into two
contexts, one without collapse_ratio and one with it.  The script reports the time of the submits that built the table
(device-resident reads, ended by a synchronise; the second context's is the warm one the collapse is compared with), rows before and after the collapse, the collapse's elapsed
time on the device stream (collapse_info, ms), and the whole finish (host clock around vfb_finish, which ends in a synchronise) with and without
collapse, twice each (the first finish of a context also takes its buffers from the allocator).

Checks: the collapsed table keeps the sum of counts, its row count is collapse_info's rows_out, and it equals
collapse_variants over the uncollapsed table.  The Python reference (tests/collapse_oracle.py) is timed on a random
sample of rows of the uncollapsed table and compared with collapse_variants on the same sample.

One JSON line per point and a summary with the card's name and power limit on stdout; --out writes the summary.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np
import pyarrow as pa
import torch

import collapse_oracle
from vfind_b200 import api

C3 = dict(seed=1003, read_len=250, adapter_len=20, region_len=198, n_variants=1000000, zipf=1, p_err=0.30, indel=0.5,
          force_indel=1, frameshift=0.05, noise=0.001, n_rate=1e-4)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def frame(offsets, data, counts):
    seq = pa.Array.from_buffers(pa.large_binary(), len(counts),
                                [None, pa.py_buffer(offsets.astype(np.int64)), pa.py_buffer(data)])
    return pa.table({"sequence": seq, "count": pa.array(counts, type=pa.uint64())})


def as_dict(tbl):
    return dict(zip(tbl.column("sequence").to_pylist(), tbl.column("count").to_pylist()))


def same_table(a, b):
    """Two (offsets, data, counts) tables hold the same rows, in any order."""
    def keyed(t):
        o, d, c = t
        raw = d.tobytes()
        return sorted((raw[int(o[i]):int(o[i + 1])], int(c[i])) for i in range(len(c)))
    return len(a[2]) == len(b[2]) and keyed(a) == keyed(b)


def build(ctx, chunks):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t, s, n in chunks:
        ctx.submit_device(t.data_ptr(), t.numel(), s.data_ptr(), n)
    ctx.sync()
    return (time.perf_counter() - t0) * 1e3


def timed_finish(ctx):
    t0 = time.perf_counter()
    out = ctx.finish_arrays(copy=True)
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", default="10000000,100000000")
    ap.add_argument("--chunk", type=int, default=12_500_000)
    ap.add_argument("--ratio", type=float, default=2.0)
    ap.add_argument("--sample", type=int, default=5000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    cfg = api.synth_cfg(**C3)
    adapters = api.synth_adapters(cfg)
    L = cfg.read_len
    points = []
    for total in [int(x) for x in args.reads.split(",")]:
        chunks, done = [], 0
        while done < total:
            n = min(args.chunk, total - done)
            t = torch.empty(n * L, dtype=torch.uint8, device=dev)
            s = torch.empty(n * 2, dtype=torch.int32, device=dev)
            api.synth_device(cfg, done, n, t.data_ptr(), s.data_ptr(), 0)
            chunks.append((t, s, n))
            done += n
        torch.cuda.synchronize()
        for skip in (False, True):
            kw = dict(device=0, batch_reads=args.chunk, table_capacity_hint=min(total, 40_000_000), skip_translation=skip)
            with api.Context(adapters, **kw) as ctx:
                build_ms = build(ctx, chunks)
                off1, plain = timed_finish(ctx)
                off2, _ = timed_finish(ctx)
            with api.Context(adapters, collapse_ratio=args.ratio, **kw) as ctx:
                build_on_ms = build(ctx, chunks)
                on1, coll = timed_finish(ctx)
                info1 = ctx.collapse_info()
                on2, coll2 = timed_finish(ctx)
                info2 = ctx.collapse_info()
            # checks at full size
            sum_ok = int(plain[2].sum(dtype=np.uint64)) == int(coll[2].sum(dtype=np.uint64))
            standalone = api.collapse_variants(frame(*plain), args.ratio)
            sa = standalone.column("sequence").combine_chunks()
            sa_tab = (np.frombuffer(sa.buffers()[1], dtype=np.int64)[:len(sa) + 1].astype(np.uint64),
                      np.frombuffer(sa.buffers()[2], dtype=np.uint8) if sa.buffers()[2] is not None else np.zeros(0, np.uint8),
                      standalone.column("count").to_numpy())
            matches = same_table(coll, sa_tab) and same_table(coll, coll2)
            # the Python reference on a random sample of rows
            rng = random.Random(total + skip)
            idx = sorted(rng.sample(range(len(plain[2])), min(args.sample, len(plain[2]))))
            o, d, c = plain
            raw = d.tobytes()
            sample = {raw[int(o[i]):int(o[i + 1])]: int(c[i]) for i in idx}
            t0 = time.perf_counter()
            want = collapse_oracle.collapse_reference(sample, args.ratio)
            ref_s = time.perf_counter() - t0
            t0 = time.perf_counter()
            got = as_dict(api.collapse_variants(pa.table({"sequence": pa.array(list(sample), pa.binary()),
                                                          "count": pa.array(list(sample.values()), pa.uint64())}), args.ratio))
            gpu_sample_s = time.perf_counter() - t0
            r = {"reads": total, "skip_translation": skip, "ratio": args.ratio,
                 # the first context of a size also pays for its warm-up; the second builds the same table warm
                 "build_ms_first_ctx": round(build_ms, 1), "build_ms_warm": round(build_on_ms, 1),
                 "rows_before": int(len(plain[2])), "rows_after": int(len(coll[2])),
                 "collapse_info": info1, "collapse_info_second": info2,
                 "finish_ms_off": [round(off1, 1), round(off2, 1)], "finish_ms_on": [round(on1, 1), round(on2, 1)],
                 "collapse_over_warm_build": round(info2["ms"] / build_on_ms, 4),
                 "finish_on_over_off": round(on2 / off2, 3),
                 "sum_kept": sum_ok, "rows_out_agrees": info1["rows_out"] == len(coll[2]),
                 "matches_standalone": matches,
                 "sample_rows": len(sample), "sample_rows_after": len(want),
                 "reference_s_on_sample": round(ref_s, 2), "standalone_call_s_on_sample": round(gpu_sample_s, 3),
                 "sample_matches_reference": got == want}
            print(json.dumps(r), flush=True)
            points.append(r)
        del chunks
        torch.cuda.empty_cache()
    ok = all(p["sum_kept"] and p["rows_out_agrees"] and p["matches_standalone"] and p["sample_matches_reference"]
             for p in points)
    summary = {"card": card(), "config": "C3, device-resident reads, one context per device", "points": points,
               "all_checks_pass": ok}
    print(json.dumps(summary), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "collapse_probe.json"), "w") as fh:
            json.dump(summary, fh, indent=1)
    if not ok:
        raise SystemExit("a check failed")


if __name__ == "__main__":
    main()
