"""Cost of umi_length on C3-shaped reads.

    python tools/umi_probe.py [--reads 100000000] [--dup-reads 12500000] [--sample 1000000] [--out DIR]

C3 reads (250-bp synthetic amplicons, 20-nt adapters, 198-nt region, 1 M library members) are generated on the device
and counted with UMIs off and with umi_length=10, umi_offset=0.  The synthetic reads start with 0-12 random lead
bases, so their first ten bytes are nearly unique: almost every read is its own molecule and the table holds about one
(variant, UMI) row per counted read.  This is close to the worst case for the table.  A second workload repeats
every span of --dup-reads reads 8 times (vfb_submit_device accepts repeated spans): 8 reads per molecule.

Per workload and mode: the step time of a cold pass and of three warm passes (host clock around the submits, ended by a
synchronise; vfb_reset before each warm pass), table rows, rows returned, and the finish twice (host clock around
vfb_finish), with the group-by's device time (umi_info ms) separately.  Both modes get the same table capacity hint,
large enough that neither grows its table: a table that grew during the cold pass keeps its larger slot array, and the
warm passes would then compare different capacities.  The sample: the first --sample reads, counted
on the device and by tests/umi_oracle.py, compared row by row.

One JSON line per point and a summary with the card's name and power limit on stdout; --out writes the summary.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np
import torch

import oracle
import umi_oracle
from vfind_b200 import api

C3 = dict(seed=1003, read_len=250, adapter_len=20, region_len=198, n_variants=1000000, zipf=1, p_err=0.30, indel=0.5,
          force_indel=1, frameshift=0.05, noise=0.001, n_rate=1e-4)
UMI = 10


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def submit_all(ctx, chunks):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t, s, n in chunks:
        ctx.submit_device(t.data_ptr(), t.numel(), s.data_ptr(), n)
    ctx.sync()
    return (time.perf_counter() - t0) * 1e3


def measure(adapters, chunks, batch, hint, umi):
    kw = dict(device=0, batch_reads=batch, table_capacity_hint=hint)
    if umi:
        kw["umi_length"] = UMI
    with api.Context(adapters, **kw) as ctx:
        cold = submit_all(ctx, chunks)
        warm = []
        for _ in range(3):
            ctx.reset()
            warm.append(round(submit_all(ctx, chunks), 1))
        st = ctx.stats()
        fin = []
        for _ in range(2):
            t0 = time.perf_counter()
            o, d, c = ctx.finish_arrays()
            fin.append(round((time.perf_counter() - t0) * 1e3, 1))
        r = {"umi_length": UMI if umi else 0, "table_capacity_hint": hint, "step_ms_cold": round(cold, 1),
             "step_ms_warm": warm, "step_ms_warm_median": sorted(warm)[1],
             "table_rows": int(st["unique"]), "rows_out": int(len(c)), "counted": int(c.sum(dtype=np.uint64)),
             "finish_ms": fin, "fused_hits": int(st["fused_hits"])}
        if umi:
            info = ctx.umi_info()
            mol = ctx.molecules()
            r.update({"group_by_ms": round(info["ms"], 2), "pairs": int(info["pairs"]), "reads_short": int(info["reads_short"]),
                      "molecules": int(mol.sum(dtype=np.uint64)), "pairs_agree": int(info["pairs"]) == int(mol.sum(dtype=np.uint64))})
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=100_000_000)
    ap.add_argument("--dup-reads", type=int, default=12_500_000)
    ap.add_argument("--chunk", type=int, default=12_500_000)
    ap.add_argument("--sample", type=int, default=1_000_000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    cfg = api.synth_cfg(**C3)
    adapters = api.synth_adapters(cfg)
    L = cfg.read_len
    points = []

    def gen(first, n):
        t = torch.empty(n * L, dtype=torch.uint8, device=dev)
        s = torch.empty(n * 2, dtype=torch.int32, device=dev)
        api.synth_device(cfg, first, n, t.data_ptr(), s.data_ptr(), 0)
        return t, s

    # the sample against the reference
    t, s = gen(0, args.sample)
    with api.Context(adapters, device=0, umi_length=UMI) as ctx:
        ctx.submit_device(t.data_ptr(), t.numel(), s.data_ptr(), args.sample)
        o, d, c = ctx.finish_arrays()
        mol = ctx.molecules()
        info = ctx.umi_info()
    raw = d.tobytes()
    got = {raw[int(o[i]):int(o[i + 1])]: (int(c[i]), int(mol[i])) for i in range(len(c))}
    text, off, ln = oracle.synth_reads(oracle.synth_cfg(**C3), 0, args.sample)
    want, short, pairs = umi_oracle.process_reads_umi(oracle.make_params(adapters), text, off, ln, UMI,
                                                      n_threads=os.cpu_count() or 1)
    sample = {"sample_reads": args.sample, "rows": len(want), "pairs": pairs, "reads_short": short,
              "matches_reference": got == want and info["pairs"] == pairs and info["reads_short"] == short}
    print(json.dumps(sample), flush=True)
    del t, s

    # C3, every read once
    chunks, done = [], 0
    while done < args.reads:
        n = min(args.chunk, args.reads - done)
        chunks.append((*gen(done, n), n))
        done += n
    torch.cuda.synchronize()
    hint = args.reads                      # room for a row per read in either mode: no table growth
    for umi in (False, True):
        r = {"workload": "C3", "reads": args.reads, **measure(adapters, chunks, args.chunk, hint, umi)}
        print(json.dumps(r), flush=True)
        points.append(r)
    del chunks
    torch.cuda.empty_cache()

    # every span of dup-reads reads repeated 8 times (8 reads per molecule), in one device batch per repeat
    t, s = gen(0, args.dup_reads)
    s8 = s.view(-1, 2).repeat(8, 1).contiguous().view(-1)
    dup = [(t, s8, 8 * args.dup_reads)]
    for umi in (False, True):
        r = {"workload": "C3 spans x8", "reads": 8 * args.dup_reads,
             **measure(adapters, dup, args.chunk, 8 * args.dup_reads, umi)}
        print(json.dumps(r), flush=True)
        points.append(r)
    ok = sample["matches_reference"] and all(p.get("pairs_agree", True) for p in points)
    summary = {"card": card(), "config": "C3, device-resident reads, one context, umi_length=%d umi_offset=0" % UMI,
               "sample": sample, "points": points, "all_checks_pass": ok}
    print(json.dumps(summary), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "umi_probe.json"), "w") as fh:
            json.dump(summary, fh, indent=1)
    if not ok:
        raise SystemExit("a check failed")


if __name__ == "__main__":
    main()
