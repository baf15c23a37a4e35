"""Context lines (ugx_find_context, ugx_find_context_batch: `-A` / `-B` / `-C`) next to the line records they start from
(ugx_find_lines, ugx_find_lines_batch) on the same device-resident inputs, in one process.

    python tools/context_bench.py [--scale 1.0] [--steps 5] [--out DIR]

Inputs (`scale` shrinks the sizes and the file count for a rehearsal; the full sizes are far larger than the 126 MB
L2):
  c2 4 GiB      -F -f words.txt            -C2, -v -C2
  c5 8 GiB      'ERROR|WARN' ...           -C2 (every line matches: no context lines, the stage's fixed cost)
  c1 4 GiB      -w the (general route)     -C2, -A5, -v -C2 (under -v the context lines need their first match)
  tree_c2       20 000 files of U(0, 4 KiB) cut from c2: find_context_batch -C2 against find_lines_batch
Times are the calls' CUDA-event times (device ms), best of `steps` after one warm-up call.  context_share is the part
of the find_context time the context stage adds over find_lines with the same flags.  Checks: the selected records
among the first 4 Mi context records are the find_lines records; for the batch, every 97th file's slice equals find_context on that file
alone.  One JSON line per input, plus the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SINGLE = [("c2", "c2", "c2", 4.0, [("C2", 2, 2, False), ("v_C2", 2, 2, True)]),
          ("c5", "c5", "c5", 8.0, [("C2", 2, 2, False)]),
          ("c1_w_the", "w_the", "c1", 4.0, [("C2", 2, 2, False), ("A5", 0, 5, False), ("v_C2", 2, 2, True)])]


def gpu_info() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as ex:  # the number is still reported, without the card's settings
        return {"gpu": "unknown (%s)" % ex}


def pattern_path(pname: str) -> str:
    p = os.path.join(ROOT, "ugrep_b200", "patterns", pname + ".ugxp")
    return p if os.path.exists(p) else os.path.join(ROOT, "tests", "golden", "patterns", pname + ".ugxp")


def best(fn, steps: int):
    """(best device ms, last totals) over `steps` calls after one warm-up call"""
    fn()
    ms, t = [], None
    for _ in range(steps):
        t = fn()
        ms.append(t.kernel_ms)
    return min(ms), t


def selected_equal(sc, n_ctx, invert, lines, k=1 << 22) -> bool:
    """the selected records among the first k records of the last context result against the find_lines records"""
    r = sc.fetch_lines(0, min(k, n_ctx))
    got = r[(r["cap"] != 0) != invert]
    return got.tobytes() == lines[:len(got)].tobytes() and (len(got) == len(lines) or len(r) == k)


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the named sizes (rehearsal)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/context_bench.jsonl")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    if not torch.cuda.is_available():
        print("context_bench: no CUDA device (the scan path has no CPU fallback)", file=sys.stderr)
        return 2
    from ugrep_b200 import api, corpus
    info = gpu_info()
    print(json.dumps(info), flush=True)
    sc = api.Scanner(0)
    rows, ok = [], True
    for name, pname, cname, gib, forms in SINGLE:
        pat = api.Pattern.load(pattern_path(pname), 0)
        block = corpus.block(cname, 32 << 20)
        reps = max(1, int(gib * args.scale * (1 << 30)) // len(block))
        dev = torch.from_numpy(block).cuda().repeat(reps)
        row = {"input": name, "gib": round(dev.numel() / (1 << 30), 2)}
        for form, b, a, inv in forms:
            lms, lt = best(lambda: sc.find_lines_device(pat, dev, invert=inv), args.steps)
            lines = sc.fetch_lines(0, min(lt.matches, 1 << 22))
            cms, ct = best(lambda: sc.find_context_device(pat, dev, b, a, invert=inv), args.steps)
            n = sc.last_lines[1]
            same = ct.matches == lt.matches and selected_equal(sc, n, inv, lines)
            ok &= same
            row[form] = {"find_lines_ms": round(lms, 3), "find_context_ms": round(cms, 3),
                         "context_ms": round(cms - lms, 3), "context_share": round((cms - lms) / cms, 3),
                         "selected": ct.matches, "printed": n, "kernel": ct.kernel, "launches": ct.launches,
                         "gbps": round(dev.numel() / cms / 1e6, 1), "identical": same}
        row.update(info)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del dev
        torch.cuda.empty_cache()

    # ---- 20 000 files in one launch sequence
    pat = api.Pattern.load(pattern_path("c2"), 0)
    base = corpus.block("c2", 8 << 20).tobytes()
    rng = np.random.default_rng(8)
    files = []
    for _ in range(max(1, int(20000 * args.scale))):
        n = int(rng.integers(0, 4097))
        lo = int(rng.integers(0, len(base) - n))
        files.append(base[lo:lo + n])
    pack, begins, lens = api._pack_files(files)
    packed = (torch.from_numpy(pack).cuda(), begins, lens)
    row = {"input": "tree_c2", "files": len(files), "mb": round(int(lens.sum()) / 1e6, 2)}
    for form, inv in (("C2", False), ("v_C2", True)):
        lms, lt = best(lambda: sc.batch_records_device(pat, packed, True, invert=inv)[1], args.steps)
        cms, ct = best(lambda: sc.find_context_batch(pat, packed, 2, 2, invert=inv)[2], args.steps)
        rec, first, _ = sc.find_context_batch(pat, packed, 2, 2, invert=inv)
        same = ct.matches == lt.matches
        for i in range(0, len(files), 97):
            one, _ = sc.find_context(pat, files[i], 2, 2, invert=inv)
            same &= rec[int(first[i]):int(first[i + 1])].tobytes() == one.tobytes()
        ok &= same
        row[form] = {"find_lines_batch_ms": round(lms, 3), "find_context_batch_ms": round(cms, 3),
                     "context_ms": round(cms - lms, 3), "context_share": round((cms - lms) / cms, 3),
                     "selected": ct.matches, "printed": len(rec), "launches": ct.launches, "identical": bool(same)}
    row.update(info)
    print(json.dumps(row), flush=True)
    rows.append(row)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "context_bench.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    if not ok:
        print("context_bench: records differ", file=sys.stderr)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
