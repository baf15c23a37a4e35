"""Boolean line queries over many files (ugx_find_lines_bool_batch, ugx_count_lines_bool_batch: `ugrep -r --and` /
`--andnot` / `--bool`, `-v`) next to the per-term batch selections they are made of and next to the two ways a caller
has without them, on device-resident batches, in one process.

    python tools/bool_batch_bench.py [--steps 5] [--loop-files 2000] [--out DIR]

Inputs: 20 000 files of U(0, 4 KiB) cut from c5 and from c2 (a source tree), and 1 000 files of 64 KiB from each; the
queries of DESIGN.md §4.4c:
  c5   ERROR --andnot 555                   [[0], [~1]]    literals
       (ERROR|WARN) --and c5                [[0, 1], [2]]  two literals and the c5 config pattern
  c2   c2 --andnot the                      [[0], [~1]]    the c2 word list and a literal
       (the|and) --and c2                   [[0, 1], [2]]  two literals and the c2 word list
each in both polarities.  The literals are compiled by the library (Pattern.literal).
Times (CUDA-event device ms, best and median of `steps` after one warm-up): terms_ms = the sum of the terms'
find_lines_batch, find_lines_bool_batch and its -v with bool_share = the part the Boolean stage adds over terms_ms,
count_lines_bool_batch.  Wall clock: loop_ms = a per-file find_lines_bool loop over the first `loop-files` files, scaled
to the whole batch; merge_ms = K find_lines_batch calls to the host (pattern 0 in both polarities, for every line's
position) plus a numpy merge.  Check: the records equal the merge, the loop's records equal their slices, and the
counts equal first[].  One JSON line per input and query, plus the card's name and power limit read in the same run.
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

QUERIES = {"c5": [("ERROR --andnot 555", [b"ERROR", b"555"], [[0], [~1]]),
                  ("(ERROR|WARN) --and c5", [b"ERROR", b"WARN", "c5"], [[0, 1], [2]])],
           "c2": [("c2 --andnot the", ["c2", b"the"], [[0], [~1]]),
                  ("(the|and) --and c2", [b"the", b"and", "c2"], [[0, 1], [2]])]}
INPUTS = [("c5", "20000 x U(0, 4 KiB)"), ("c2", "20000 x U(0, 4 KiB)"), ("c5", "1000 x 64 KiB"),
          ("c2", "1000 x 64 KiB")]


def gpu_info() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as ex:  # the number is still reported, without the card's settings
        return {"gpu": "unknown (%s)" % ex}


def make_files(cname: str, shape: str, corpus) -> list:
    base = corpus.block(cname, 8 << 20).tobytes()
    rng = np.random.default_rng(20000 if shape.startswith("20000") else 1000)
    files = []
    if shape.startswith("20000"):
        for _ in range(20000):
            lo = int(rng.integers(0, len(base) - 4096))
            files.append(base[lo:lo + int(rng.integers(0, 4097))])
    else:
        for _ in range(1000):
            lo = int(rng.integers(0, len(base) - 65536))
            files.append(base[lo:lo + 65536])
    return files


def timed(fn, steps: int):
    """(best device ms, median device ms, last result) over `steps` calls after one warm-up call"""
    fn()
    ms, r = [], None
    for _ in range(steps):
        r = fn()
        ms.append((r[-1] if isinstance(r, tuple) else r).kernel_ms)
    return min(ms), statistics.median(ms), r


def host_merge(sc, pats, cnf, src, invert, line_dtype):
    """the caller's alternative: every term's batch line records to the host (pattern 0 in both polarities gives every
    line of every file), then a numpy merge over the batch's lines numbered across the files"""
    hit0, f_hit, _ = sc.find_lines_batch(pats[0], src)
    miss0, f_miss, _ = sc.find_lines_batch(pats[0], src, invert=True)
    per_file = np.diff(f_hit.astype(np.int64)) + np.diff(f_miss.astype(np.int64))
    lb = np.zeros(len(per_file) + 1, dtype=np.int64)
    lb[1:] = np.cumsum(per_file)

    def gidx(rec, first):
        fid = np.repeat(np.arange(len(per_file)), np.diff(first.astype(np.int64)))
        return lb[fid] + rec["line"].astype(np.int64) - 1

    every = np.empty(int(lb[-1]), dtype=line_dtype)
    masks = np.zeros(int(lb[-1]), dtype=np.uint32)
    g = gidx(hit0, f_hit)
    every[g] = hit0
    masks[g] |= np.uint32(1)
    every[gidx(miss0, f_miss)] = miss0
    for j in range(1, len(pats)):
        hit, f, _ = sc.find_lines_batch(pats[j], src)
        masks[gidx(hit, f)] |= np.uint32(1 << j)
    ok = np.ones(len(masks), dtype=bool)
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
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--loop-files", type=int, default=2000, help="files of the per-file find_lines_bool loop")
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/bool_batch_bench.jsonl")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    if not torch.cuda.is_available():
        print("bool_batch_bench: no CUDA device (the scan path has no CPU fallback)", file=sys.stderr)
        return 2
    from ugrep_b200 import api, corpus
    info = gpu_info()
    print(json.dumps(info), flush=True)
    sc = api.Scanner(0)
    rows, ok = [], True
    for cname, shape in INPUTS:
        files = make_files(cname, shape, corpus)
        pack, begins, lens = api._pack_files(files)
        dev = torch.from_numpy(pack).cuda()
        src = (dev, begins, lens)
        for qname, terms, cnf in QUERIES[cname]:
            pats = [api.Pattern.load(os.path.join(ROOT, "ugrep_b200", "patterns", t + ".ugxp"), 0)
                    if isinstance(t, str) else api.Pattern.literal(t, 0) for t in terms]
            terms_ms = sum(timed(lambda: sc.batch_records_device(p, src, True), args.steps)[0] for p in pats)
            row = {"input": cname, "files": shape, "mib": round(sum(map(len, files)) / (1 << 20), 1), "query": qname,
                   "cnf": cnf, "terms_ms": round(terms_ms, 3)}
            for form, inv in (("plain", False), ("v", True)):
                fb, fm, (first, ft) = timed(lambda: sc.find_lines_bool_batch_device(pats, cnf, src, inv), args.steps)
                cb, cm, (counts, ct) = timed(lambda: sc.count_lines_bool_batch(pats, cnf, src, inv), args.steps)
                first, ft = sc.find_lines_bool_batch_device(pats, cnf, src, inv)
                got = sc.fetch_lines(0, ft.matches)
                t0 = time.perf_counter()
                want = host_merge(sc, pats, cnf, src, inv, api.LINE_DTYPE)
                merge_ms = (time.perf_counter() - t0) * 1e3
                nloop = min(args.loop_files, len(files))
                loop = []
                t0 = time.perf_counter()
                for i in range(nloop):
                    b = int(begins[i])
                    loop.append(sc.find_lines_bool(pats, cnf, dev[b:b + len(files[i])], inv)[0])
                loop_ms = (time.perf_counter() - t0) * 1e3 * len(files) / nloop
                same = (got.tobytes() == want.tobytes() and ct.matches == ft.matches == len(want)
                        and np.array_equal(counts, np.diff(first.astype(np.int64)).astype(np.uint64))
                        and all(got[int(first[i]):int(first[i + 1])].tobytes() == loop[i].tobytes()
                                for i in range(nloop)))
                ok &= same
                row[form] = {"find_lines_bool_batch_ms": round(fb, 3), "find_lines_bool_batch_median_ms": round(fm, 3),
                             "count_lines_bool_batch_ms": round(cb, 3),
                             "count_lines_bool_batch_median_ms": round(cm, 3),
                             "bool_share": round((fb - terms_ms) / fb, 3), "loop_ms": round(loop_ms, 1),
                             "merge_ms": round(merge_ms, 1), "selected": ft.matches, "newlines": ft.newlines,
                             "launches": ft.launches, "identical": bool(same)}
                del got, want, loop
            row.update(info)
            print(json.dumps(row), flush=True)
            rows.append(row)
        del dev
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bool_batch_bench.jsonl"), "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    if not ok:
        print("bool_batch_bench: records differ between the forms", file=sys.stderr)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
