"""Cost of both_strands on the C3 shape with device-resident reads.

    python tools/strand_probe.py [--reads 100000000] [--steps 3] [--out DIR]

100 M reads per step (C3: 250-bp synthetic merged amplicon reads, 20-nt adapters, 30 % of adapters mutated) are
generated on the device.  A torch kernel then reverse-complements a fraction f of the fixed-length reads in place
(every 1/f-th read), which stands for a library ligated in no fixed direction.  For f in {0, 0.5} and both_strands
off / on the script reports ms per step, reads/s, reverse_reads and reverse_counted, with the card's name and power
limit.  Each table of a 1 M-read sample is checked against the oracle (tests/strand_oracle.py with both_strands,
oracle.process_reads without).  One JSON line per point, and the summary, on stdout.
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
import strand_oracle
from vfind_b200 import api

C3 = dict(seed=1003, read_len=250, adapter_len=20, region_len=198, n_variants=1000000, zipf=1, p_err=0.30, indel=0.5,
          force_indel=1, frameshift=0.05, noise=0.001, n_rate=1e-4)
THR = 0.75


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def rc_every(t: torch.Tensor, n: int, L: int, f: float):
    """Reverse-complement reads 0, k, 2k, ... (k = round(1/f)) of a fixed-stride text in place."""
    if f <= 0:
        return
    k = int(round(1 / f))
    lut = torch.arange(256, dtype=torch.uint8, device=t.device)
    lut[torch.tensor(list(b"ACGTUacgtu"), device=t.device).long()] = torch.tensor(list(b"TGCAAtgcaa"), dtype=torch.uint8,
                                                                                   device=t.device)
    rows = t.view(n, L)[::k]
    for i in range(0, rows.shape[0], 1 << 20):
        part = rows[i:i + (1 << 20)]
        part.copy_(lut[part.long()].flip(1))


def table_dict(offsets, data, counts):
    raw = data.tobytes()
    return {raw[int(offsets[i]):int(offsets[i + 1])]: int(counts[i]) for i in range(len(counts))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=100_000_000)
    ap.add_argument("--chunk", type=int, default=12_500_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sample", type=int, default=1_000_000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    cfg = api.synth_cfg(**C3)
    adapters = api.synth_adapters(cfg)
    L = cfg.read_len
    chunks = []
    done = 0
    while done < args.reads:
        n = min(args.chunk, args.reads - done)
        t = torch.empty(n * L, dtype=torch.uint8, device=dev)
        s = torch.empty(n * 2, dtype=torch.int32, device=dev)
        api.synth_device(cfg, done, n, t.data_ptr(), s.data_ptr(), 0)
        chunks.append((t, s, n))
        done += n
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)
    p = oracle.make_params(adapters, accept_prefix_alignment=THR, accept_suffix_alignment=THR)
    results = []
    applied = 0.0
    for f in (0.0, 0.5):
        if f != applied:
            for t, _, n in chunks:
                rc_every(t, n, L, f)
            torch.cuda.synchronize()
            applied = f
        # the oracle's view of the first `sample` reads of this input
        st_, ss_ = chunks[0][0], chunks[0][1]
        m = min(args.sample, chunks[0][2])
        h_text = st_[:m * L].cpu().numpy()
        h_sp = ss_[:2 * m].cpu().numpy().view(np.uint32).reshape(m, 2)
        for both in (False, True):
            t0 = time.perf_counter()
            if both:
                want = strand_oracle.process_reads_both_strands(p, h_text, h_sp[:, 0], h_sp[:, 1], n_threads=os.cpu_count() or 8)[0]
            else:
                want = oracle.process_reads(p, h_text, h_sp[:, 0], h_sp[:, 1], n_threads=os.cpu_count() or 8)[0]
            oracle_s = time.perf_counter() - t0
            with api.Context(adapters, device=0, batch_reads=args.chunk, table_capacity_hint=min(args.reads, 40_000_000),
                             accept_prefix_alignment=THR, accept_suffix_alignment=THR, both_strands=both) as ctx:
                ctx.set_compute_stream(stream.cuda_stream)
                ctx.submit_device(st_.data_ptr(), m * L, ss_.data_ptr(), m)
                sample_ok = table_dict(*ctx.finish_arrays()) == want
                with torch.cuda.stream(stream):
                    for _ in range(args.warmup):
                        ctx.table_clear()
                        for t, s, n in chunks:
                            ctx.submit_device(t.data_ptr(), t.numel(), s.data_ptr(), n)
                    ctx.fence()
                    stream.synchronize()
                    ctx.reset()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for _ in range(args.steps):
                        ctx.table_clear()
                        for t, s, n in chunks:
                            ctx.submit_device(t.data_ptr(), t.numel(), s.data_ptr(), n)
                    ctx.fence()
                    e1.record(stream)
                    stream.synchronize()
                ms = e0.elapsed_time(e1) / args.steps
                st = ctx.stats()
            r = {"f": f, "both_strands": both, "ms_per_step": round(ms, 3), "reads_per_s": args.reads / (ms * 1e-3),
                 "reverse_reads_per_step": st["reverse_reads"] // args.steps,
                 "reverse_counted_per_step": st["reverse_counted"] // args.steps,
                 "counted_per_step": st["counted"] // args.steps,
                 "sample_reads": m, "sample_matches_oracle": sample_ok, "oracle_s": round(oracle_s, 1)}
            print(json.dumps(r), flush=True)
            results.append(r)
    base = {r["f"]: r["ms_per_step"] for r in results if not r["both_strands"]}
    summary = {"card": card(), "reads_per_step": args.reads, "steps": args.steps, "config": "C3, device-resident",
               "points": results,
               "on_over_off": {str(r["f"]): round(r["ms_per_step"] / base[r["f"]], 4) for r in results if r["both_strands"]},
               "on_f05_over_on_f0": round([r["ms_per_step"] for r in results if r["both_strands"] and r["f"] == 0.5][0] /
                                          [r["ms_per_step"] for r in results if r["both_strands"] and r["f"] == 0.0][0], 4),
               "all_samples_match": all(r["sample_matches_oracle"] for r in results)}
    print(json.dumps(summary), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "strand_probe.json"), "w") as fh:
            json.dump(summary, fh, indent=1)
    if not summary["all_samples_match"]:
        raise SystemExit("a sample table differs from the oracle")


if __name__ == "__main__":
    main()
