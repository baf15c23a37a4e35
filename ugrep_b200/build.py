"""Build libugrep_b200.so in-tree with nvcc for sm_100a (B200).

    python -m ugrep_b200.build [--force] [--verbose]

The library is the product: hand-written CUDA kernels + the C ABI of
include/ugrep_b200.h.  It is built next to this file so that it travels to the
GPU box with the repository snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libugrep_b200.so")
SOURCES = ["capi.cu", "scan_kernels.cu", "line_records.cu", "records_kernel.cu", "match_lines.cu", "span_scan.cu", "newline_count.cu", "utf8_check.cu", "batch_kernel.cu", "batch_records.cu", "context_lines.cu", "bool_lines.cu", "fast_kernels.cu", "stream_count.cu", "stream_literal.cu", "stream_search.cu", "pattern_host.cpp", "sharded.cpp", "literal_compile.cpp", "wordlist_compile.cpp"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the scan path is CUDA-only and cannot be built without it")


def newest_source() -> float:
    t = 0.0
    for root, _, files in os.walk(CSRC):
        for f in files:
            t = max(t, os.path.getmtime(os.path.join(root, f)))
    t = max(t, os.path.getmtime(os.path.join(HERE, "..", "include", "ugrep_b200.h")))
    return t


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= newest_source():
        return LIB
    # one nvcc per translation unit, in parallel (objects under build/, git-ignored), then one link
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = ["-O3", "-std=c++17", "-lineinfo", *ARCH, "-Xcompiler", "-fPIC,-O2,-Wall"]
    if verbose:
        flags += ["-Xptxas", "-v"]

    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".hpp", ".h", ".inc"))]
    headers.append(os.path.join(HERE, "..", "include", "ugrep_b200.h"))
    headers.append(os.path.abspath(__file__))
    hdr_time = max(os.path.getmtime(h) for h in headers)

    def compile_one(src: str):
        obj = os.path.join(objdir, os.path.splitext(src)[0] + (".v.o" if verbose else ".o"))
        if (not force and os.path.exists(obj)
                and os.path.getmtime(obj) >= max(hdr_time, os.path.getmtime(os.path.join(CSRC, src)))):
            return src, obj, subprocess.CompletedProcess([], 0, "", "(up to date)")
        cmd = [nvcc(), *flags, "-c", "-o", obj, os.path.join(CSRC, src)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    objs = []
    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        for src, obj, r in ex.map(compile_one, SOURCES):
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError("nvcc failed on " + src)
            if verbose:
                print("==", src)
                print(r.stdout + r.stderr)
            objs.append(obj)
    r = subprocess.run([nvcc(), *ARCH, "-shared", "-o", LIB, *objs, "-lcudart"], capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
