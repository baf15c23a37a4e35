"""Line records (ugx_find_lines) next to count_lines and find_all_device on the same buffers, in one process.

    python tools/lines_bench.py [--scale 1.0] [--steps 5] [--out DIR]

Inputs (resident in HBM, CUDA-event timed; `scale` shrinks them for a rehearsal):
  c2   ugrep -F -f words.txt            4 GiB   span route
  c5   -e 'ERROR|WARN' -e '\\d{3}-\\d{4}'  8 GiB   span route
  c3b  [A-Z][a-z]+ing on the c3 corpus  4 GiB   span route
  w    -w the (META, line-at-a-time)    4 GiB of the c1 corpus
For each: count_lines, find_all_device, find_lines and find_lines -v (kernel time = the call's device time, and the
wall time of the call); then end to end from a page-locked host buffer INCLUDING the copy of the records to the host
(find_lines into a host array).  Checks: the first 8 MiB block against the oracle (both polarities), and at full size
matching == count_lines and matching + inverted == lines.  One JSON line per input, plus the card's name and power
limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

INPUTS = [("c2", os.path.join("ugrep_b200", "patterns", "c2.ugxp"), "c2", 4.0),
          ("c5", os.path.join("ugrep_b200", "patterns", "c5.ugxp"), "c5", 8.0),
          ("c3b", os.path.join("ugrep_b200", "patterns", "c3b.ugxp"), "c3", 4.0),
          ("w_the", os.path.join("tests", "golden", "patterns", "w_the.ugxp"), "c1", 4.0)]
BLOCK = 32 << 20


def gpu_info() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as ex:  # the number is still reported, without the card's settings
        return {"gpu": "unknown (%s)" % ex}


def timed(fn, steps: int):
    """(best device ms reported by the call, best wall ms) over `steps` calls after one warm-up call"""
    fn()
    dev, wall = [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        t = fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(t.kernel_ms)
    return min(dev), min(wall), t


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the named sizes (rehearsal)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/lines_bench.jsonl")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("lines_bench: no CUDA device (the scan path has no CPU fallback)", file=sys.stderr)
        return 2
    from ugrep_b200 import api, corpus
    import lines_oracle as LO
    info = gpu_info()
    print(json.dumps(info), flush=True)
    sc = api.Scanner(0)
    rows = []
    for name, rel, cname, gib in INPUTS:
        path = os.path.join(ROOT, rel)
        pat = api.Pattern.load(path, 0)
        op = LO.oracle(path)
        block = corpus.block(cname, BLOCK)
        reps = max(1, int(gib * args.scale * (1 << 30)) // len(block))
        dev = torch.from_numpy(block).cuda().repeat(reps)
        n = dev.numel()
        # ---- checks: a block against the oracle, consistency at full size
        head = block[:8 << 20]
        cut = int(np.flatnonzero(head == 10)[-1]) + 1
        head = head[:cut]
        for inv in (False, True):
            rec, _ = sc.find_lines(pat, torch.from_numpy(head).cuda(), invert=inv)
            if rec.tobytes() != op.find_lines(head, invert=inv).tobytes():
                print("lines_bench: %s invert=%s differs from the oracle" % (name, inv), file=sys.stderr)
                return 1
        lines = reps * int((block == 10).sum())
        row = {"input": name, "gib": round(n / (1 << 30), 3)}
        ms, wall, t = timed(lambda: sc.count_lines(pat, dev), args.steps)
        row["count_lines"] = {"ms": round(ms, 3), "wall_ms": round(wall, 3), "gbps": round(n / ms / 1e6, 1), "kernel": t.kernel,
                              "count": t.matches}
        count = t.matches
        ms, wall, t = timed(lambda: sc.find_all_device(pat, dev), args.steps)
        row["find_all_device"] = {"ms": round(ms, 3), "wall_ms": round(wall, 3), "gbps": round(n / ms / 1e6, 1),
                                  "kernel": t.kernel, "records": t.matches}
        got = {}
        for inv in (False, True):
            ms, wall, t = timed(lambda: sc.find_lines_device(pat, dev, invert=inv), args.steps)
            got[inv] = t.matches
            row["find_lines" + ("_v" if inv else "")] = {"ms": round(ms, 3), "wall_ms": round(wall, 3),
                                                        "gbps": round(n / ms / 1e6, 1), "kernel": t.kernel,
                                                        "records": t.matches, "handover": bool(t.flags & 2)}
        if got[False] != count or got[False] + got[True] != lines:
            print("lines_bench: %s: %d matching lines, count_lines %d, %d inverted, %d lines"
                  % (name, got[False], count, got[True], lines), file=sys.stderr)
            return 1
        # ---- end to end from page-locked memory, records copied to the host
        host = dev.cpu().pin_memory()
        hp = host.numpy()
        for inv in (False, True):
            sc.find_lines(pat, hp, invert=inv)
            best = None
            for _ in range(max(1, args.steps // 2)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rec, t = sc.find_lines(pat, hp, invert=inv)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            row["e2e_pinned" + ("_v" if inv else "")] = {"s": round(best, 4), "gbps": round(n / best / 1e9, 2),
                                                         "records": len(rec), "record_mb": round(rec.nbytes / 1e6, 1)}
            del rec
        row.update(info)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del dev, host, hp
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "lines_bench.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
