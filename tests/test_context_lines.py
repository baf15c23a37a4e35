"""Context lines (ugx_find_context*, `ugrep -n -A/-B/-C`) on the CPU: the declarations in the header and the ctypes
signatures, and the oracle's derivation (context_oracle.py) pinned on hand-written cases."""
import os
import re

import numpy as np
import pytest

import context_oracle as CO
import golden_lib as G
import lines_oracle as LO
import oracle_lib as O

HEADER = os.path.join(O.ROOT, "include", "ugrep_b200.h")
M = CO.UINT32_MAX


def declaration(name):
    text = open(HEADER).read()
    m = re.search(r"int\s+%s\s*\(([^;]*)\);" % name, text)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def test_context_declarations():
    one = ["ugx_scanner *s", "const ugx_pattern *p", "const void *buf", "uint64_t nbytes", "uint64_t base_offset",
           "uint64_t base_line", "uint32_t flags", "uint32_t before", "uint32_t after"]
    assert declaration("ugx_find_context_device") == one + ["const ugx_line **dev_out", "uint64_t *n_out",
                                                            "ugx_totals *totals"]
    assert declaration("ugx_find_context") == one + ["ugx_line *out", "uint64_t cap", "uint64_t *n_out",
                                                     "ugx_totals *totals"]
    assert declaration("ugx_find_context_batch") == [
        "ugx_scanner *s", "const ugx_pattern *p", "const void *buf", "uint64_t nbytes", "const uint64_t *begins",
        "const uint64_t *lens", "uint64_t nfiles", "uint32_t flags", "uint32_t before", "uint32_t after",
        "uint64_t *first", "ugx_line *out", "uint64_t cap", "uint64_t *n_out", "ugx_totals *totals"]
    assert "#define UGX_ABI_VERSION 2" in open(HEADER).read()


def test_ctypes_signatures():
    import ctypes as C
    from ugrep_b200 import api
    L = api.lib()
    u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
    one = [vp, vp, vp, u64, u64, u64, u32, u32, u32]
    assert L.ugx_find_context.argtypes == one + [vp, u64, C.POINTER(u64), C.POINTER(api._Totals)]
    assert L.ugx_find_context_device.argtypes == one + [C.POINTER(vp), C.POINTER(u64), C.POINTER(api._Totals)]
    assert L.ugx_find_context_batch.argtypes == [vp, vp, vp, u64, vp, vp, u64, u32, u32, u32, vp, vp, u64,
                                                 C.POINTER(u64), C.POINTER(api._Totals)]
    assert {"ugx_find_context", "ugx_find_context_device", "ugx_find_context_batch"} <= set(api.EXPORTS)


@pytest.mark.parametrize("n, sel, b, a, want", [
    (10, [3, 5], 1, 1, [2, 3, 4, 5, 6]),          # overlapping windows
    (10, [2, 5], 1, 1, [1, 2, 3, 4, 5, 6]),       # adjacent windows (3 and 4 touch)
    (10, [2, 6], 1, 1, [1, 2, 3, 5, 6, 7]),       # a gap of exactly one line (4)
    (10, [1], 5, 0, [0, 1]),                      # before reaching past line 1
    (10, [8], 0, 5, [8, 9]),                      # after reaching past the last line
    (10, [0, 9], 0, 0, [0, 9]),                   # no context: the selected lines
    (10, [4], 2, 3, [2, 3, 4, 5, 6, 7]),
    (1, [0], M, M, [0]),
    (7, [3], M, M, list(range(7))),               # one selected line, unbounded windows: every line
    (7, [], M, M, []),
])
def test_printed_lines(n, sel, b, a, want):
    assert list(CO.printed(n, sel, b, a)) == want


def lines_of(rec):
    return [int(x) for x in rec["line"]]


@pytest.fixture(scope="module")
def op():
    return LO.oracle(G.pattern_path("c1"))


H = b"Sherlock Holmes"


def test_hand_written_buffers(op):
    body = [b"a", H, b"b", b"c", b"", b"d", H + b" x", b"e", b"f", b"g", b"h", H]
    for tail in (b"\n", b""):
        data = b"\n".join(body) + tail
        assert lines_of(op.find_lines(data)) == [2, 7, 12]
        assert lines_of(CO.find_context(op, data, 0, 0)) == [2, 7, 12]
        assert lines_of(CO.find_context(op, data, 1, 1)) == [1, 2, 3, 6, 7, 8, 11, 12]
        assert lines_of(CO.find_context(op, data, 2, 2)) == [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12]
        assert lines_of(CO.find_context(op, data, 0, 4)) == [2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12]
        assert lines_of(CO.find_context(op, data, 3, 0)) == [1, 2, 4, 5, 6, 7, 9, 10, 11, 12]
        assert lines_of(CO.find_context(op, data, M, M)) == list(range(1, 13))
        # -v: the non-matching lines are selected, the matching ones are context
        v = CO.find_context(op, data, 0, 1, invert=True)
        assert lines_of(v) == list(range(1, 13))
        sel = CO.is_selected(v, True)
        assert [int(r["line"]) for r, s in zip(v, sel) if not s] == [2, 7, 12]
        for r in v:
            if int(r["line"]) in (2, 7, 12):
                assert int(r["cap"]) != 0 and int(r["offset"]) == int(r["bol"])
            else:
                assert (int(r["cap"]), int(r["len"]), int(r["offset"])) == (0, 0, int(r["bol"]))
        # every record is the one find_lines gives that line in its own polarity
        both = {int(r["line"]): r.tobytes() for r in np.concatenate([op.find_lines(data), op.find_lines(data, True)])}
        for r in CO.find_context(op, data, 2, 3):
            assert r.tobytes() == both[int(r["line"])]


def test_empty_lines_and_empty_buffer(op):
    assert len(CO.find_context(op, b"", M, M)) == 0
    assert len(CO.find_context(op, b"", M, M, invert=True)) == 0
    assert lines_of(CO.find_context(op, b"\n\n\n", 1, 1)) == []
    assert lines_of(CO.find_context(op, b"\n\n\n", 1, 1, invert=True)) == [1, 2, 3]
    data = b"\n\n" + H + b"\n\n\n"
    r = CO.find_context(op, data, 1, 1)
    assert [(int(x["line"]), int(x["bol"]), int(x["eol"])) for x in r] == [(2, 1, 1), (3, 2, 17), (4, 18, 18)]


def test_bases_move_lines_and_offsets(op):
    data = b"x\n" + H + b"\ny\nz"
    base_line = (1 << 64) - (1 << 33)
    r = CO.find_context(op, data, M, M, base_offset=1 << 33, base_line=base_line)
    assert lines_of(r) == [base_line + k for k in (1, 2, 3, 4)]
    assert int(r["bol"][0]) == 1 << 33
