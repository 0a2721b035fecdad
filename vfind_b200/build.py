"""Builds vfind_b200/libvfind_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch).

    python -m vfind_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libvfind_b200.so")
OBJ = os.path.join(HERE, "_obj")
SOURCES = ["api.cu", "multi.cu", "ingest.cu", "pgunzip.cu", "gunzip_gpu.cu", "kernels_parse.cu", "kernels_inflate.cu", "kernels_scan.cu", "kernels_dp.cu", "kernels_dpw.cu", "kernels_count.cu", "kernels_misc.cu", "kernels_strand.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xptxas", "-v"]


CXX = os.environ.get("CXX", "g++")


def _obj_name(src):
    return os.path.splitext(src)[0] + ".o"


def _deps():
    hdr = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdr.append(os.path.join(os.path.dirname(HERE), "include", "vfind_b200.h"))
    return hdr


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdr = _deps()
    jobs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, _obj_name(s))
        if force or _stale(obj, [src] + hdr):
            jobs.append((src, obj))

    def cc(job):
        src, obj = job
        if src.endswith(".cpp"):      # host-only code: g++
            cmd = [CXX, "-O3", "-std=c++17", "-fPIC", "-Wall", "-c", src, "-o", obj]
        else:
            cmd = [NVCC] + FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = r.stdout + r.stderr
        with open(obj + ".log", "w") as f:
            f.write(log)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, log))
        return log

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            logs = list(ex.map(cc, jobs))
        if verbose:
            for l in logs:
                print(l)
    objs = [os.path.join(OBJ, _obj_name(s)) for s in SOURCES]
    if force or jobs or _stale(OUT, objs):
        r = subprocess.run([NVCC, "-shared", "-o", OUT] + objs + ["-lz", "-cudart", "static",
                                                                    "-gencode", "arch=compute_100a,code=sm_100a"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return OUT


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
