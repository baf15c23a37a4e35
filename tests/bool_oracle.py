"""The oracle of Boolean line queries (`ugrep -e A --and -e B`, `--andnot`, `--bool`, ugx_find_lines_bool): a derivation
from the oracle's line records (lines_oracle.py) that does not depend on how the library divides the work.

TEST INFRASTRUCTURE.
1. Pattern 0's matching and non-matching line records together are every line of the buffer, each exactly once.
2. M(L), the term mask of a line: bit j is set iff L is one of pattern j's matching records.
3. A line satisfies the query iff every clause (pos, neg) has (M & pos) != 0 or (~M & neg) != 0; the selected lines
   are those that do (with invert, those that do not).  Each keeps bol / eol, with offset = bol, len = 0, cap = M.
"""
from __future__ import annotations

import numpy as np


def pairs(cnf) -> list[tuple[int, int]]:
    """(pos, neg) bit masks of a CNF written as lists of ints (j = pattern j matches, ~j = it does not)"""
    out = []
    for clause in cnf:
        pos = neg = 0
        for t in clause:
            if t >= 0:
                pos |= 1 << t
            else:
                neg |= 1 << ~t
        out.append((pos, neg))
    return out


def every_line(op0, data, base_offset: int = 0, base_line: int = 0) -> np.ndarray:
    """every line of the buffer as a record, from pattern 0's matching and non-matching records"""
    every = np.concatenate([op0.find_lines(data, False, base_offset, base_line),
                            op0.find_lines(data, True, base_offset, base_line)])
    every = every[np.argsort(every["line"], kind="stable")]
    want = np.arange(base_line + 1, base_line + 1 + len(every), dtype=np.uint64)
    assert np.array_equal(every["line"], want), "matching and non-matching lines are not lines 1..N exactly once"
    return every


def term_masks(ops, data, nlines: int, base_offset: int = 0, base_line: int = 0) -> np.ndarray:
    """M(L) of every line (0-based)"""
    m = np.zeros(nlines, dtype=np.uint32)
    for j, op in enumerate(ops):
        hit = op.find_lines(data, False, base_offset, base_line)
        m[(hit["line"] - np.uint64(base_line) - np.uint64(1)).astype(np.int64)] |= np.uint32(1 << j)
    return m


def satisfies(masks: np.ndarray, clauses) -> np.ndarray:
    """which lines satisfy the conjunction of (pos, neg) clauses"""
    ok = np.ones(len(masks), dtype=bool)
    for pos, neg in clauses:
        ok &= ((masks & np.uint32(pos)) != 0) | ((~masks & np.uint32(neg)) != 0)
    return ok


def find_lines_bool(ops, cnf, data, invert: bool = False, base_offset: int = 0, base_line: int = 0) -> np.ndarray:
    """the records ugx_find_lines_bool should return; ops[j] has find_lines (lines_oracle.oracle), cnf is a CNF of
    int lists or a list of (pos, neg) pairs"""
    clauses = [c if isinstance(c, tuple) else pairs([c])[0] for c in cnf]
    every = every_line(ops[0], data, base_offset, base_line)
    masks = term_masks(ops, data, len(every), base_offset, base_line)
    sel = satisfies(masks, clauses) != invert
    rec = every[sel].copy()
    rec["offset"] = rec["bol"]
    rec["len"] = 0
    rec["cap"] = masks[sel]
    return rec
