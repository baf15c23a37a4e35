"""Boolean line queries (ugx_find_lines_bool, ugx_count_lines_bool: `--and` / `--andnot` / `--bool`, `-v`) next to the
per-term line selections they are made of, and next to the host alternative, on device-resident inputs, in one process.

    python tools/bool_bench.py [--scale 1.0] [--steps 5] [--out DIR]

Inputs (`scale` shrinks the sizes for a rehearsal; the full sizes are far larger than the 126 MB L2):
  c5 8 GiB   ERROR --andnot 555                   [[0], [~1]]    literals
             (ERROR|WARN) --and c5                [[0, 1], [2]]  two literals and the c5 config pattern
  c2 4 GiB   c2 --andnot the                      [[0], [~1]]    the c2 word list and a literal
             (the|and) --and c2                   [[0, 1], [2]]  two literals and the c2 word list
each in both polarities.  The literals are compiled by the library (Pattern.literal).
Times: find_lines_bool and count_lines_bool as CUDA-event device ms (best and median of `steps` after one warm-up);
terms_ms = the sum of the terms' find_lines device ms (best of each), bool_share = the part of find_lines_bool the
Boolean stage adds over the terms' selections; host_ms = wall clock of the alternative a caller has without the stage:
find_lines of every term to the host (pattern 0 in both polarities, for every line's position) plus a numpy merge.
Check: the records equal that host merge.  One JSON line per input and query, plus the card's name and power limit
read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

INPUTS = [("c5", 8.0, [("ERROR --andnot 555", [b"ERROR", b"555"], [[0], [~1]]),
                       ("(ERROR|WARN) --and c5", [b"ERROR", b"WARN", "c5"], [[0, 1], [2]])]),
          ("c2", 4.0, [("c2 --andnot the", ["c2", b"the"], [[0], [~1]]),
                       ("(the|and) --and c2", [b"the", b"and", "c2"], [[0, 1], [2]])])]


def gpu_info() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as ex:  # the number is still reported, without the card's settings
        return {"gpu": "unknown (%s)" % ex}


def timed(fn, steps: int):
    """(best device ms, median device ms, last totals) over `steps` calls after one warm-up call"""
    fn()
    ms, t = [], None
    for _ in range(steps):
        t = fn()
        ms.append(t.kernel_ms)
    return min(ms), statistics.median(ms), t


def host_merge(sc, pats, cnf, dev, invert, line_dtype):
    """the host alternative: every term's matching lines to the host, pattern 0's other lines too, then numpy"""
    hit0, _ = sc.find_lines(pats[0], dev)
    miss0, _ = sc.find_lines(pats[0], dev, invert=True)
    nlines = len(hit0) + len(miss0)
    every = np.empty(nlines, dtype=line_dtype)
    every[(hit0["line"] - 1).astype(np.int64)] = hit0
    every[(miss0["line"] - 1).astype(np.int64)] = miss0
    masks = np.zeros(nlines, dtype=np.uint32)
    masks[(hit0["line"] - 1).astype(np.int64)] |= np.uint32(1)
    del hit0, miss0
    for j in range(1, len(pats)):
        hit, _ = sc.find_lines(pats[j], dev)
        masks[(hit["line"] - 1).astype(np.int64)] |= np.uint32(1 << j)
        del hit
    ok = np.ones(nlines, dtype=bool)
    for clause in cnf:
        pos = sum(1 << t for t in clause if t >= 0)
        neg = sum(1 << ~t for t in clause if t < 0)
        ok &= ((masks & np.uint32(pos)) != 0) | ((~masks & np.uint32(neg)) != 0)
    sel = ok != invert
    rec = every[sel]
    rec["offset"] = rec["bol"]
    rec["len"] = 0
    rec["cap"] = masks[sel]
    return rec


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the named sizes (rehearsal)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/bool_bench.jsonl")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    if not torch.cuda.is_available():
        print("bool_bench: no CUDA device (the scan path has no CPU fallback)", file=sys.stderr)
        return 2
    from ugrep_b200 import api, corpus
    info = gpu_info()
    print(json.dumps(info), flush=True)
    sc = api.Scanner(0)
    rows, ok = [], True
    for cname, gib, queries in INPUTS:
        block = corpus.block(cname, 32 << 20)
        reps = max(1, int(gib * args.scale * (1 << 30)) // len(block))
        dev = torch.from_numpy(block).cuda().repeat(reps)
        for qname, terms, cnf in queries:
            pats = [api.Pattern.load(os.path.join(ROOT, "ugrep_b200", "patterns", t + ".ugxp"), 0)
                    if isinstance(t, str) else api.Pattern.literal(t, 0) for t in terms]
            terms_ms = sum(timed(lambda: sc.find_lines_device(p, dev), args.steps)[0] for p in pats)
            row = {"input": cname, "gib": round(dev.numel() / (1 << 30), 2), "query": qname, "cnf": cnf,
                   "terms_ms": round(terms_ms, 3)}
            t0 = time.perf_counter()
            want = host_merge(sc, pats, cnf, dev, False, api.LINE_DTYPE)
            host_ms = (time.perf_counter() - t0) * 1e3
            for form, inv in (("plain", False), ("v", True)):
                fb, fm, ft = timed(lambda: sc.find_lines_bool_device(pats, cnf, dev, invert=inv), args.steps)
                cb, cm, ctot = timed(lambda: sc.count_lines_bool(pats, cnf, dev, invert=inv), args.steps)
                sc.find_lines_bool_device(pats, cnf, dev, invert=inv)
                got = sc.fetch_lines(0, sc.last_lines[1])
                if inv:
                    want = host_merge(sc, pats, cnf, dev, True, api.LINE_DTYPE)
                same = got.tobytes() == want.tobytes() and ctot.matches == len(want) == ft.matches
                ok &= same
                row[form] = {"find_lines_bool_ms": round(fb, 3), "find_lines_bool_median_ms": round(fm, 3),
                             "count_lines_bool_ms": round(cb, 3), "count_lines_bool_median_ms": round(cm, 3),
                             "bool_share": round((fb - terms_ms) / fb, 3), "selected": ft.matches,
                             "newlines": ft.newlines, "launches": ft.launches, "identical": bool(same)}
                del got
            row["host_ms"] = round(host_ms, 1)
            row.update(info)
            print(json.dumps(row), flush=True)
            rows.append(row)
            del want
        del dev
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bool_bench.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    if not ok:
        print("bool_bench: records differ from the host merge", file=sys.stderr)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
