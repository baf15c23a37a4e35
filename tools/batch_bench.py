"""Records of many files in one launch sequence (ugx_find_lines_batch, ugx_find_all_batch) next to ugx_count_batch and
a per-file loop over the same packed buffer, in one process.

    python tools/batch_bench.py [--scale 1.0] [--steps 5] [--out DIR]

Inputs (packed on 16-byte boundaries and resident in HBM; `scale` shrinks the file counts for a rehearsal):
  tree_c5   20 000 files of U(0, 4 KiB) cut from the c5 corpus, -e 'ERROR|WARN' -e '\\d{3}-\\d{4}'
  tree_c2   20 000 files of U(0, 4 KiB) cut from the c2 corpus, -F -f words.txt
  big_c5     1 000 files of 64 KiB cut from the c5 corpus
For each: find_lines_batch, find_lines_batch -v, find_all_batch and count_batch (device ms = the call's CUDA-event
time, wall ms = the call including its host synchronises; best of `steps`), and the per-file loop of find_lines,
find_lines -v and find_all_device over device views of the same buffer (no host-to-device copy; records left on the
device; one pass, device ms = the sum of the calls' event times).  files/s and GB/s are over the files' bytes.
Check: the batch records equal the per-file records of every file, in all three forms.  One JSON line per input,
plus the card's name and power limit read in the same run.
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

INPUTS = [("tree_c5", "c5", "c5", 20000, None), ("tree_c2", "c2", "c2", 20000, None), ("big_c5", "c5", "c5", 1000, 65536)]


def gpu_info() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as ex:  # the number is still reported, without the card's settings
        return {"gpu": "unknown (%s)" % ex}


def make_files(cname: str, count: int, size: int | None, seed: int = 8):
    from ugrep_b200 import corpus
    base = corpus.block(cname, 4 << 20).tobytes()
    rng = np.random.default_rng(seed)
    files = []
    for _ in range(count):
        n = size if size is not None else int(rng.integers(0, 4096))
        lo = int(rng.integers(0, len(base) - n))
        files.append(base[lo:lo + n])
    return files


def timed(fn, steps: int):
    """(best device ms reported by the call, best wall ms, last result) over `steps` calls after one warm-up call"""
    fn()
    dev, wall = [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        r = fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append((r[1] if isinstance(r, tuple) else r).kernel_ms)
    return min(dev), min(wall), r


def rates(ms: float, wall: float, nfiles: int, nbytes: int) -> dict:
    return {"ms": round(ms, 3), "wall_ms": round(wall, 3), "files_per_s": round(nfiles / wall * 1e3),
            "gbps": round(nbytes / ms / 1e6, 2), "gbps_wall": round(nbytes / wall / 1e6, 2)}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the named file counts (rehearsal)")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/batch_bench.jsonl")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    if not torch.cuda.is_available():
        print("batch_bench: no CUDA device (the scan path has no CPU fallback)", file=sys.stderr)
        return 2
    from ugrep_b200 import api
    info = gpu_info()
    print(json.dumps(info), flush=True)
    sc = api.Scanner(0)
    rows = []
    for name, pname, cname, count, size in INPUTS:
        pat = api.Pattern.load(os.path.join(ROOT, "ugrep_b200", "patterns", pname + ".ugxp"), 0)
        files = make_files(cname, max(1, int(count * args.scale)), size)
        pack, begins, lens = api._pack_files(files)
        dev = torch.from_numpy(pack).cuda()
        packed = (dev, begins, lens)
        nfiles, nbytes = len(files), int(lens.sum())
        views = [dev[int(b):int(b) + int(n)] for b, n in zip(begins, lens)]
        row = {"input": name, "files": nfiles, "mb": round(nbytes / 1e6, 2)}

        # ---- one launch sequence for all files
        forms = {"find_lines_batch": lambda: sc.batch_records_device(pat, packed, True),
                 "find_lines_batch_v": lambda: sc.batch_records_device(pat, packed, True, invert=True),
                 "find_all_batch": lambda: sc.batch_records_device(pat, packed, False)}
        batch = {}
        for form, fn in forms.items():
            ms, wall, (first, t) = timed(fn, args.steps)
            row[form] = dict(rates(ms, wall, nfiles, nbytes), records=t.matches, launches=t.launches, kernel=t.kernel)
            rec = sc.fetch(0, t.matches) if form == "find_all_batch" else sc.fetch_lines(0, t.matches)
            batch[form] = (first, rec)
        ms, wall, (counts, t) = timed(lambda: sc.count_batch(pat, packed, "matches"), args.steps)
        row["count_batch"] = dict(rates(ms, wall, nfiles, nbytes), count=t.matches, launches=t.launches)

        # ---- one call per file over device views of the same buffer
        loops = {"find_lines_batch": lambda v: sc.find_lines_device(pat, v),
                 "find_lines_batch_v": lambda v: sc.find_lines_device(pat, v, invert=True),
                 "find_all_batch": lambda v: sc.find_all_device(pat, v)}
        same = True
        for form, call in loops.items():
            call(views[0])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dms = 0.0
            for v in views:
                dms += call(v).kernel_ms
            wall = (time.perf_counter() - t0) * 1e3
            row[form.replace("_batch", "_per_file")] = rates(dms, wall, nfiles, nbytes)
            # untimed: every file's records from its own call against its slice of the batch
            first, rec = batch[form]
            for i, v in enumerate(views):
                t = call(v)
                got = sc.fetch(0, t.matches) if form == "find_all_batch" else sc.fetch_lines(0, t.matches)
                if got.tobytes() != rec[int(first[i]):int(first[i + 1])].tobytes():
                    print("batch_bench: %s %s file %d differs from its own call" % (name, form, i), file=sys.stderr)
                    same = False
                    break
        row["identical"] = same
        for form in forms:
            row[form]["speedup_vs_per_file"] = round(row[form.replace("_batch", "_per_file")]["wall_ms"] / row[form]["wall_ms"], 1)
        row.update(info)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del dev, views, packed
        torch.cuda.empty_cache()
        if not same:
            return 1
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "batch_bench.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
