"""`-c` through the search automaton (count_lines_search_kernel) against the same call with the scanner option
"no_search" (count_lines_stream_kernel alone), on the same device-resident inputs, in one process.

    python tools/search_bench.py [--scale 1.0] [--steps 10] [--out DIR]

Inputs (tiled from a seeded line-aligned 32 MiB block; `scale` shrinks them for a rehearsal; the full sizes are far
larger than the 126 MB L2):
  c2    4 GiB   -F -f words.txt (1,000 words, the dense corpus)
  c2s   4 GiB   the same words, the sparse corpus
  c4    8 GiB   the Greek word list
  w3000 4 GiB   3,000 words from tools/big_list.py (its automaton is refused by size: both calls take today's kernel)
The two routes alternate call by call.  Times are the calls' CUDA-event times (device ms): best and median of `steps`
after one warm-up call each, with the spread (max - min) / median.  The counts of both routes must agree with each
other and with the block's oracle count times the tiling.  One JSON line per input, plus the card's name and power
limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

INPUTS = [("c2", "c2", 4.0), ("c2s", "c2", 4.0), ("c4", "c4", 8.0), ("w3000", None, 4.0)]


def gpu_info() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as ex:  # the number is still reported, without the card's settings
        return {"gpu": "unknown (%s)" % ex}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("search_bench.py: no CUDA device")
    from ugrep_b200 import api, corpus
    import oracle_lib as O
    info = gpu_info()
    print(json.dumps(info), flush=True)
    rows = []
    with tempfile.TemporaryDirectory() as tmp:
        for name, pname, gib in INPUTS:
            if pname is None:
                opc, pf = api.compile_words(corpus.words_list(11, 3000))
                path = os.path.join(tmp, "w3000.ugxp")
                api.write_ugxp(path, opc, pf)
                cname = "c2"
            else:
                path = os.path.join(ROOT, "ugrep_b200", "patterns", pname + ".ugxp")
                cname = name
            block = corpus.block(cname, 32 << 20)
            reps = max(1, int(gib * a.scale * (1 << 30)) // len(block))
            want = reps * O.OraclePattern(path).count_lines(block)
            dev = torch.from_numpy(block).cuda().repeat(reps)
            pat = api.Pattern.load(path, 0)
            scs = {"search": api.Scanner(0), "no_search": api.Scanner(0)}
            scs["no_search"].set_option("no_search", 1)
            ms = {k: [] for k in scs}
            tot = {}
            for k, sc in scs.items():
                sc.count_lines(pat, dev)
            for _ in range(a.steps):
                for k, sc in scs.items():
                    t = sc.count_lines(pat, dev)
                    ms[k].append(t.kernel_ms)
                    tot[k] = t
            for k in scs:
                if tot[k].matches != want:
                    raise SystemExit("search_bench.py: %s %s counted %d, want %d" % (name, k, tot[k].matches, want))
            nbytes = dev.numel()
            row = {"input": name, "bytes": nbytes, "lines": want, **info}
            for k in scs:
                v = np.array(ms[k])
                med = float(np.median(v))
                row[k] = {"kernel": tot[k].kernel, "launches": tot[k].launches, "best_ms": round(float(v.min()), 3),
                          "median_ms": round(med, 3), "spread": round(float((v.max() - v.min()) / med), 4),
                          "GBps_best": round(nbytes / (v.min() * 1e-3) / 1e9, 1)}
            row["speedup_best"] = round(row["no_search"]["best_ms"] / row["search"]["best_ms"], 3)
            print(json.dumps(row), flush=True)
            rows.append(row)
            del dev
            torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "search_bench.json"), "w") as f:
            json.dump({"card": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
