"""Line records (ugx_find_lines, `ugrep -c` / `ugrep -v` per line) on the CPU: the oracle's line records (tests/oracle_lines.c) against the
committed golden fixtures made with the unmodified reference, the partition of the lines into matching and
non-matching ones, and the ABI's declaration of the new entry points."""
import os
import re

import numpy as np
import pytest

import golden_lib as G
import lines_oracle as LO
import oracle_lib as O

HEADER = os.path.join(O.ROOT, "include", "ugrep_b200.h")


def text_lines(data: bytes):
    """(bol, eol) of every line: a buffer that ends in '\\n' has no empty line after it"""
    out, bol = [], 0
    for i, b in enumerate(data):
        if b == 0x0A:
            out.append((bol, i))
            bol = i + 1
    if bol < len(data):
        out.append((bol, len(data)))
    return out


@pytest.mark.parametrize("name", G.pattern_names())
def test_find_lines_vs_golden(name):
    op = LO.oracle(G.pattern_path(name))
    for case, data in G.cases(name):
        rec = op.find_lines(data)
        assert len(rec) == case["lines"], (name, case["input"])
        lines = text_lines(data)
        for r in rec:
            assert (int(r["bol"]), int(r["eol"])) == lines[int(r["line"]) - 1], (name, case["input"], r)
            assert r["bol"] <= r["offset"] <= r["eol"] and r["cap"] != 0
        # the first match record per line of `ugrep -n -b -o` (the golden list, as the oracle's find_all restates it)
        allm = op.find_all(data)
        G.check_list(case, data, allm)
        first = {}
        for m in allm:
            first.setdefault(int(m["line"]), m)
        if "list" in case:
            want_lines = sorted({int(ln.split(b":", 1)[0]) for ln in G.base64.b64decode(case["list"]).split(b"\n") if ln})
            assert sorted(set(int(x) for x in rec["line"])) == want_lines, (name, case["input"])
        got = [(int(r["line"]), int(r["offset"]), int(r["len"]), int(r["cap"])) for r in rec]
        want = [(ln, int(m["offset"]), int(m["len"]), int(m["cap"])) for ln, m in sorted(first.items())]
        assert got == want, (name, case["input"])


@pytest.mark.parametrize("name", G.pattern_names())
def test_inverted_and_matching_lines_partition_the_lines(name):
    op = LO.oracle(G.pattern_path(name))
    for case, data in G.cases(name):
        lines = text_lines(data)
        hit = op.find_lines(data)
        miss = op.find_lines(data, invert=True)
        nums = sorted([int(x) for x in hit["line"]] + [int(x) for x in miss["line"]])
        assert nums == list(range(1, len(lines) + 1)), (name, case["input"])
        assert len(lines) == O.newlines(data) + (1 if data and data[-1:] != b"\n" else 0)
        for r in miss:
            bol, eol = lines[int(r["line"]) - 1]
            assert (int(r["bol"]), int(r["eol"]), int(r["offset"]), int(r["len"]), int(r["cap"])) == (bol, eol, bol, 0, 0)
        # bases move every line number and offset
        shifted = op.find_lines(data, invert=True, base_offset=1 << 33, base_line=1 << 32)
        assert np.array_equal(shifted["line"], miss["line"] + (1 << 32))
        assert np.array_equal(shifted["bol"], miss["bol"] + (1 << 33))


def test_edge_buffers():
    op = LO.oracle(G.pattern_path("c1"))
    assert len(op.find_lines(b"")) == 0 and len(op.find_lines(b"", invert=True)) == 0
    r = op.find_lines(b"\n", invert=True)
    assert [(int(x["line"]), int(x["bol"]), int(x["eol"])) for x in r] == [(1, 0, 0)]
    data = b"a Sherlock Holmes\r\nxyz\r\nSherlock Holmes"
    hit = op.find_lines(data)
    assert [(int(x["line"]), int(x["bol"]), int(x["eol"]), int(x["offset"])) for x in hit] == [(1, 0, 18, 2), (3, 24, 39, 24)]
    miss = op.find_lines(data, invert=True)
    assert [(int(x["line"]), int(x["bol"]), int(x["eol"])) for x in miss] == [(2, 19, 23)]


def test_header_declares_line_records():
    text = open(HEADER).read()
    for sym in ("ugx_find_lines", "ugx_find_lines_device", "ugx_scanner_fetch_lines", "ugx_sharded_find_lines"):
        assert re.search(r"\b%s\s*\(" % sym, text), sym
    assert "UGX_LINES_INVERT 1u" in text and "UGX_K_SPAN_LINES = 10" in text
    from ugrep_b200 import api
    assert {"ugx_find_lines", "ugx_find_lines_device", "ugx_scanner_fetch_lines", "ugx_sharded_find_lines"} <= set(api.EXPORTS)
    assert api.LINE_DTYPE.itemsize == 40 and LO.LINE_DTYPE == api.LINE_DTYPE


def test_sizeof_ugx_line_is_40(tmp_path):
    """the C compiler's view of the struct (offsets included) matches LINE_DTYPE"""
    import shutil
    import subprocess
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "s.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "ugrep_b200.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu\\n",'
                   ' sizeof(ugx_line), offsetof(ugx_line, line), offsetof(ugx_line, bol), offsetof(ugx_line, eol),'
                   ' offsetof(ugx_line, offset), offsetof(ugx_line, len), offsetof(ugx_line, cap)); return 0;}\n')
    exe = tmp_path / "s"
    subprocess.run([cc, "-I" + os.path.join(O.ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    from ugrep_b200 import api
    want = [api.LINE_DTYPE.itemsize] + [api.LINE_DTYPE.fields[f][1] for f in ("line", "bol", "eol", "offset", "len", "cap")]
    assert [int(x) for x in out] == want == [40, 0, 8, 16, 24, 32, 36]
