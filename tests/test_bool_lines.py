"""Boolean line queries (ugx_*_lines_bool, `--and` / `--andnot` / `--bool`) on the CPU: the declarations in the header
and the ctypes signatures, api.bool_clauses, and the oracle's derivation (bool_oracle.py) pinned by its identities on
every golden pattern's cases."""
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


def declaration(name):
    text = open(HEADER).read()
    m = re.search(r"int\s+%s\s*\(([^;]*)\);" % name, text)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def test_bool_declarations():
    query = ["ugx_scanner *s", "const ugx_pattern *const *patterns", "uint32_t npatterns",
             "const ugx_bool_clause *clauses", "uint32_t nclauses", "const void *buf", "uint64_t nbytes"]
    assert declaration("ugx_count_lines_bool") == query + ["uint32_t flags", "ugx_totals *totals"]
    one = query + ["uint64_t base_offset", "uint64_t base_line", "uint32_t flags"]
    assert declaration("ugx_find_lines_bool_device") == one + ["const ugx_line **dev_out", "uint64_t *n_out",
                                                               "ugx_totals *totals"]
    assert declaration("ugx_find_lines_bool") == one + ["ugx_line *out", "uint64_t cap", "uint64_t *n_out",
                                                        "ugx_totals *totals"]
    text = open(HEADER).read()
    assert "#define UGX_ABI_VERSION 2" in text
    assert "#define UGX_BOOL_MAX_PATTERNS 32" in text and "#define UGX_BOOL_MAX_CLAUSES  64" in text
    assert "UGX_K_BOOL_LINES = 12" in text


def test_ctypes_signatures():
    from ugrep_b200 import api
    L = api.lib()
    u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
    query = [vp, vp, u32, vp, u32, vp, u64]
    assert L.ugx_count_lines_bool.argtypes == query + [u32, C.POINTER(api._Totals)]
    assert L.ugx_find_lines_bool_device.argtypes == query + [u64, u64, u32, C.POINTER(vp), C.POINTER(u64),
                                                             C.POINTER(api._Totals)]
    assert L.ugx_find_lines_bool.argtypes == query + [u64, u64, u32, vp, u64, C.POINTER(u64), C.POINTER(api._Totals)]
    assert {"ugx_count_lines_bool", "ugx_find_lines_bool", "ugx_find_lines_bool_device"} <= set(api.EXPORTS)
    assert C.sizeof(api.BoolClause) == 8
    assert L.ugx_kernel_name(12) == b"bool_count_kernel"


def as_pairs(arr):
    return [(c.pos, c.neg) for c in arr]


def test_bool_clauses_conversions():
    from ugrep_b200 import api
    assert as_pairs(api.bool_clauses([[0], [1]])) == [(1, 0), (2, 0)]                  # -e A --and -e B
    assert as_pairs(api.bool_clauses([[0], [~1]])) == [(1, 0), (0, 2)]                 # A --andnot B
    assert as_pairs(api.bool_clauses([[0, 1], [~2]])) == [(3, 0), (0, 4)]              # --bool 'A|B -C'
    assert as_pairs(api.bool_clauses([[~0]])) == [(0, 1)]                              # --not A
    assert as_pairs(api.bool_clauses([[0, ~0], (31, ~31, 3)])) == [(1, 1), ((1 << 31) | 8, 1 << 31)]
    assert as_pairs(api.bool_clauses([[np.int64(2), 2]])) == [(4, 0)]
    assert len(api.bool_clauses([])) == 0
    assert len(api.bool_clauses([[0]] * 65)) == 65  # the clause limit is the library's to enforce
    assert as_pairs(api.bool_clauses([[0, 1], [~2]])) == BO.pairs([[0, 1], [~2]])


@pytest.mark.parametrize("cnf", [None, 0, "0", [0], [[]], [[0], []], [[32]], [[~32]], [[1.0]], [[True]], [["a"]],
                                 [[0], None], {0: [0]}])
def test_bool_clauses_rejects_malformed_cnfs(cnf):
    from ugrep_b200 import api
    with pytest.raises(ValueError):
        api.bool_clauses(cnf)


def lines_of(rec):
    return [int(x) for x in rec["line"]]


H = b"Sherlock Holmes"


def test_hand_written_query():
    a, b = LO.oracle(G.pattern_path("c1")), LO.oracle(G.pattern_path("w_the"))
    body = [b"a", H, b"the " + H, b"the", b"", H + b" the", b"x"]
    for tail in (b"\n", b""):
        data = b"\n".join(body) + tail
        assert lines_of(BO.find_lines_bool([a, b], [[0], [1]], data)) == [3, 6]
        assert lines_of(BO.find_lines_bool([a, b], [[0], [~1]], data)) == [2]
        assert lines_of(BO.find_lines_bool([a, b], [[0, 1]], data)) == [2, 3, 4, 6]
        assert lines_of(BO.find_lines_bool([a, b], [[0, 1]], data, invert=True)) == [1, 5, 7]
        rec = BO.find_lines_bool([a, b], [], data, base_offset=1 << 33, base_line=1 << 40)
        assert lines_of(rec) == [(1 << 40) + k for k in range(1, 8)]
        assert [int(x) for x in rec["cap"]] == [0, 1, 3, 2, 0, 3, 0]
        assert (rec["offset"] == rec["bol"]).all() and not rec["len"].any() and int(rec["bol"][0]) == 1 << 33
    assert len(BO.find_lines_bool([a, b], [], b"")) == 0
    assert lines_of(BO.find_lines_bool([a, b], [[~0]], b"\n\n")) == [1, 2]


def records_of(rec):
    return np.stack([rec["line"], rec["bol"], rec["eol"]], axis=1).tobytes()


@pytest.mark.parametrize("name", G.pattern_names())
def test_derivation_identities(name):
    """on every golden case of the pattern A (B = another golden pattern): {pos=A} = A's matching lines, {neg=A} = A's
    -v lines, {pos=A},{neg=A} = nothing, {pos=A,neg=A} = every line, -v of {pos=A},{pos=B} = {neg=A|B}, no clause =
    every line"""
    names = G.pattern_names()
    other = names[(names.index(name) + 1) % len(names)]
    A, B = LO.oracle(G.pattern_path(name)), LO.oracle(G.pattern_path(other))
    for _, data in G.cases(name):
        hit, miss = A.find_lines(data), A.find_lines(data, True)
        every = BO.every_line(A, data)
        q = lambda cnf, inv=False: BO.find_lines_bool([A, B], cnf, data, inv)  # noqa: E731
        assert records_of(q([[0]])) == records_of(hit)
        assert (q([[0]])["cap"] & 1).all()
        assert records_of(q([[~0]])) == records_of(miss)
        assert records_of(q([[0]], True)) == records_of(miss)
        assert len(q([[0], [~0]])) == 0
        assert records_of(q([[0, ~0]])) == records_of(every) == records_of(q([]))
        assert q([[0], [1]], True).tobytes() == q([[~0, ~1]]).tobytes()
        assert len(q([], True)) == 0
