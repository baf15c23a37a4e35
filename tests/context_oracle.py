"""The oracle of context lines (`ugrep -n -A/-B/-C`, ugx_find_context): a derivation from the oracle's line records
(lines_oracle.py) that does not depend on how the library divides the work.

TEST INFRASTRUCTURE.
1. The matching and the non-matching line records together are every line of the buffer, each exactly once.
2. A line is printed when it lies within [s - before, s + after] of a selected line s (the matching lines, or with
   invert the non-matching ones); windows stop at the buffer's first and last line.  Every printed line keeps the
   record of its own polarity.
"""
from __future__ import annotations

import numpy as np

UINT32_MAX = (1 << 32) - 1


def printed(nlines: int, selected, before: int, after: int) -> np.ndarray:
    """0-based indices of the printed lines of a buffer of `nlines` lines, `selected` the 0-based selected lines"""
    diff = np.zeros(nlines + 1, dtype=np.int64)
    for s in selected:
        s = int(s)
        diff[max(0, s - before)] += 1
        diff[min(nlines - 1, s + after) + 1] -= 1
    return np.nonzero(np.cumsum(diff[:nlines]) > 0)[0]


def find_context(op, data, before: int, after: int, invert: bool = False, base_offset: int = 0,
                 base_line: int = 0) -> np.ndarray:
    """the records ugx_find_context should return, from op.find_lines (lines_oracle.oracle)"""
    hit = op.find_lines(data, False, base_offset, base_line)
    miss = op.find_lines(data, True, base_offset, base_line)
    every = np.concatenate([hit, miss])
    every = every[np.argsort(every["line"], kind="stable")]
    nlines = len(every)
    want = np.arange(base_line + 1, base_line + 1 + nlines, dtype=np.uint64)
    assert np.array_equal(every["line"], want), "matching and non-matching lines are not lines 1..N exactly once"
    sel = miss if invert else hit
    idx = printed(nlines, (sel["line"] - np.uint64(base_line) - np.uint64(1)).astype(np.int64), before, after)
    return every[idx]


def is_selected(rec: np.ndarray, invert: bool) -> np.ndarray:
    """the caller's rule: a record is a selected line iff (cap != 0) != invert, otherwise a context line"""
    return (rec["cap"] != 0) != invert
