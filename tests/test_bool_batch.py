"""Boolean line queries over many files (ugx_count_lines_bool_batch / ugx_find_lines_bool_batch, `ugrep -r --and`) on
the CPU: the declarations in the header and the ctypes signatures, and the per-file derivation of the expected result
(find_lines_bool_batch below, which test_bool_batch_gpu.py shares) on every golden pattern's cases: each file's slice
is the file's own Boolean result, first[] comes from the per-file lengths, and counts are those lengths."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import bool_oracle as BO
import golden_lib as G
import lines_oracle as LO
import oracle_lib as O

HEADER = os.path.join(O.ROOT, "include", "ugrep_b200.h")


def find_lines_bool_batch(ops, cnf, files, invert: bool = False):
    """(records, first, counts) that ugx_find_lines_bool_batch / ugx_count_lines_bool_batch should return for a list of
    files: bool_oracle.find_lines_bool on every file alone (bases 0), concatenated in file order; file i owns
    records[first[i]:first[i + 1]], and counts[i] = first[i + 1] - first[i]"""
    per = [BO.find_lines_bool(ops, cnf, f, invert) for f in files]
    counts = np.array([len(r) for r in per], dtype=np.uint64)
    first = np.zeros(len(files) + 1, dtype=np.uint64)
    first[1:] = np.cumsum(counts, dtype=np.uint64)
    from ugrep_b200.api import LINE_DTYPE
    records = np.concatenate(per) if per else np.zeros(0, dtype=LINE_DTYPE)
    return records, first, counts


EDGE = [b"", b"\n", b"\n\n\n", b"x", b"Sherlock Holmes", b"Sherlock Holmes\n", b"a\r\nSherlock Holmes\r\n\r\nb\r\n", b""]


def declaration(name):
    text = open(HEADER).read()
    m = re.search(r"int\s+%s\s*\(([^;]*)\);" % name, text)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def test_bool_batch_declarations():
    query = ["ugx_scanner *s", "const ugx_pattern *const *patterns", "uint32_t npatterns",
             "const ugx_bool_clause *clauses", "uint32_t nclauses", "const void *buf", "uint64_t nbytes",
             "const uint64_t *begins", "const uint64_t *lens", "uint64_t nfiles", "uint32_t flags"]
    assert declaration("ugx_count_lines_bool_batch") == query + ["uint64_t *counts", "ugx_totals *totals"]
    assert declaration("ugx_find_lines_bool_batch") == query + ["uint64_t *first", "ugx_line *out", "uint64_t cap",
                                                               "uint64_t *n_out", "ugx_totals *totals"]
    assert "#define UGX_ABI_VERSION 2" in open(HEADER).read()


def test_ctypes_signatures():
    from ugrep_b200 import api
    L = api.lib()
    u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
    query = [vp, vp, u32, vp, u32, vp, u64, vp, vp, u64, u32]
    assert L.ugx_count_lines_bool_batch.argtypes == query + [vp, C.POINTER(api._Totals)]
    assert L.ugx_find_lines_bool_batch.argtypes == query + [vp, vp, u64, C.POINTER(u64), C.POINTER(api._Totals)]
    assert {"ugx_count_lines_bool_batch", "ugx_find_lines_bool_batch"} <= set(api.EXPORTS)
    for m in ("count_lines_bool_batch", "find_lines_bool_batch", "find_lines_bool_batch_device"):
        assert callable(getattr(api.Scanner, m)), m


def records_of(rec):
    return np.stack([rec["line"], rec["bol"], rec["eol"]], axis=1).tobytes()


@pytest.mark.parametrize("name", G.pattern_names())
def test_per_file_derivation(name):
    """the batch expectation on the pattern's golden cases plus edge files (empty ones first, among and last): every
    file's slice is find_lines_bool of that file alone, first[] is the prefix of the lengths, counts are the lengths,
    and the two polarities split every file's lines"""
    names = G.pattern_names()
    other = names[(names.index(name) + 1) % len(names)]
    A, B = LO.oracle(G.pattern_path(name)), LO.oracle(G.pattern_path(other))
    files = [b""] + [data for _, data in G.cases(name)] + EDGE
    for cnf in ([[0], [1]], [[0], [~1]], [[0, 1]], [[~0]], []):
        for inv in (False, True):
            rec, first, counts = find_lines_bool_batch([A, B], cnf, files, inv)
            assert len(first) == len(files) + 1 and int(first[0]) == 0 and int(first[-1]) == len(rec)
            assert np.array_equal(np.diff(first.astype(np.int64)), counts.astype(np.int64))
            for i, f in enumerate(files):
                want = BO.find_lines_bool([A, B], cnf, f, inv)
                assert rec[int(first[i]):int(first[i + 1])].tobytes() == want.tobytes(), (name, cnf, inv, i)
                assert int(counts[i]) == len(want)
            if not inv:
                _, _, neg = find_lines_bool_batch([A, B], cnf, files, True)
                lines = [f.count(b"\n") + (1 if f and not f.endswith(b"\n") else 0) for f in files]
                assert list(map(int, counts + neg)) == lines, (name, cnf)
    # {pos=A} per file is A's matching lines of that file; an empty file selects nothing in either polarity
    rec, first, counts = find_lines_bool_batch([A, B], [[0]], files)
    for i, f in enumerate(files):
        assert records_of(rec[int(first[i]):int(first[i + 1])]) == records_of(A.find_lines(f)), (name, i)
    for inv in (False, True):
        assert int(find_lines_bool_batch([A, B], [], [b""], inv)[2][0]) == 0
    rec, first, counts = find_lines_bool_batch([A, B], [[0]], [])
    assert len(rec) == 0 and list(first) == [0] and len(counts) == 0
