"""CPU-side checks of the batch record entry points (ugx_find_all_batch, ugx_find_lines_batch): their declarations in
the header, and the packing of a list of files that the Python forms share with count_batch."""
import os
import re

import numpy as np

import oracle_lib as O

HEADER = os.path.join(O.ROOT, "include", "ugrep_b200.h")


def declaration(name):
    text = open(HEADER).read()
    m = re.search(r"int\s+%s\s*\(([^;]*)\);" % name, text)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def test_batch_record_declarations():
    common = ["ugx_scanner *s", "const ugx_pattern *p", "const void *buf", "uint64_t nbytes", "const uint64_t *begins",
              "const uint64_t *lens", "uint64_t nfiles"]
    assert declaration("ugx_find_all_batch") == common + ["uint64_t *first", "ugx_match *out", "uint64_t cap",
                                                          "uint64_t *n_out", "ugx_totals *totals"]
    assert declaration("ugx_find_lines_batch") == common + ["uint32_t flags", "uint64_t *first", "ugx_line *out",
                                                            "uint64_t cap", "uint64_t *n_out", "ugx_totals *totals"]
    assert "#define UGX_ABI_VERSION 2" in open(HEADER).read()


def test_files_are_packed_on_16_byte_boundaries():
    from ugrep_b200 import api
    files = [b"", b"abc\n", b"x" * 16, b"y" * 17, b"", b"z"]
    pack, begins, lens = api._pack_files(files)
    assert list(begins) == [0, 0, 16, 32, 64, 64] and list(lens) == [0, 4, 16, 17, 0, 1]
    assert pack.size == 80 and pack.dtype == np.uint8
    for b, f in zip(begins, files):
        assert pack[int(b):int(b) + len(f)].tobytes() == f
    assert pack[4:16].tobytes() == b"X" * 12 and pack[49:64].tobytes() == b"X" * 15
    pack, begins, lens = api._pack_files([])
    assert pack.size == 16 and len(begins) == len(lens) == 0
