"""CPU model of the shared-memory wavefronts of count_lines_search_kernel (csrc/stream_search.cu): lanes run the search
automaton of `ugx_search_describe` over stretches of S bytes, each from the empty set D - 1 bytes before its start, and
for every warp-level LDS (class map, transition) the model counts the distinct 32-bit words requested in the most
loaded of the 32 banks.  It also reports how many lane-bytes sit in MATCHED (row 0, read as a broadcast).  Not a
measurement: it sizes a layout before it is built.

    python tools/search_smem_model.py [c2 c2s c4] [--stretch 64,256,512]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_search_dfa as T  # noqa: E402
from ugrep_b200 import corpus  # noqa: E402


def wavefronts(words):
    """words: (steps, 32) word addresses of one warp-level load per row"""
    return sum(int(np.bincount(np.unique(w) % 32, minlength=32).max()) for w in words)


def model(cfg, stretch, nbytes=1 << 21):
    info, cls, table = T.describe(os.path.join(ROOT, "ugrep_b200", "patterns", ("c2" if cfg == "c2s" else cfg) + ".ugxp"))
    a = corpus.block(cfg, 8 << 20)[:nbytes]
    d1 = info.depth - 1
    ncls = info.classes
    cw = tw = steps = nmatched = 0
    for base in range(0, nbytes - 32 * stretch + 1, 4 * 32 * stretch):   # every 4th group of 32 stretches
        lanes = []
        for lane in range(32):
            s0 = base + lane * stretch
            lo = max(0, s0 - d1)
            lanes.append(np.concatenate([np.full(d1 - (s0 - lo), 10, np.uint8), a[lo:s0 + stretch]]))
        L = np.stack(lanes)
        st = np.full(32, ncls, np.int64)
        cwords, twords = [], []
        for i in range(L.shape[1]):
            c = cls[L[:, i]]
            cwords.append(L[:, i].astype(np.int64) >> 2)
            twords.append((2 * (st + c)) >> 2)     # the table starts at a 512-byte boundary
            st = table[st + c]
            if i >= d1:
                nmatched += int((st == 0).sum())
        cw += wavefronts(np.array(cwords))
        tw += wavefronts(np.array(twords))
        steps += L.shape[1]
    payload = steps * stretch / (stretch + d1)
    print("%-4s D=%d states=%d classes=%d S=%d: per warp-step cls %.2f trans %.2f wavefronts; per payload warp-byte %.2f;"
          " MATCHED %.2f of lane-bytes" % (cfg, info.depth, info.states, ncls, stretch, cw / steps, tw / steps,
                                           (cw + tw) / payload, nmatched / (payload * 32)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=["c2", "c2s", "c4"])
    ap.add_argument("--stretch", default="64,256,512")
    a = ap.parse_args()
    for cfg in a.configs:
        for s in (int(x) for x in a.stretch.split(",")):
            model(cfg, s)


if __name__ == "__main__":
    main()
