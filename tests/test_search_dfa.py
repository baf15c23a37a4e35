"""CPU test of the line-resetting search automaton of `-c` (csrc/pattern_host.cpp build_search_dfa, run on the device by
count_lines_search_kernel in csrc/stream_search.cu) through the host-only entry point ugx_search_describe.

The automaton is run here in numpy exactly as a lane runs it: from the empty set, D - 1 bytes before each position
(the buffer's start reads as '\\n'), one class lookup and one transition per byte, success = state offset 0.  A line
counts iff it holds a success; the count must be the oracle's `ugrep -c` count."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

import golden_lib as G
import oracle_lib as O
from ugrep_b200 import corpus

LIB = os.path.join(O.ROOT, "ugrep_b200", "libugrep_b200.so")
CONFIGS = sorted(glob.glob(os.path.join(O.ROOT, "ugrep_b200", "patterns", "*.ugxp")))
OK, META, ACC0, CYCLE, DEPTH, NEWLINE, SIZE, ROUTE = range(8)


class SearchInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("eligible", "refusal", "depth", "states", "classes", "table_bytes")]


def load_ugxp(path):
    import struct
    b = open(path, "rb").read()
    nop, _, pf_size, flags = struct.unpack_from("<4I", b, 8)
    return b[24 + pf_size:24 + pf_size + 4 * nop], nop, b[24:24 + pf_size], flags


def describe(path):
    lib = C.CDLL(LIB)
    lib.ugx_last_error.restype = C.c_char_p
    opc, nop, pf, flags = load_ugxp(path)
    info = SearchInfo()
    cls = (C.c_uint8 * 256)()
    table = (C.c_uint16 * 65536)()
    rc = lib.ugx_search_describe(opc, nop, pf, flags, C.byref(info), cls, table, 65536)
    assert rc == 0, lib.ugx_last_error()
    n = info.states * info.classes
    return info, np.frombuffer(cls, dtype=np.uint8).astype(np.int64), np.frombuffer(table, dtype=np.uint16)[:n].astype(np.int64)


def lane_states(info, cls, table, a, skip=None):
    """state after each byte, each computed from the empty set D - 1 bytes before it (skip: warm-up length)"""
    w = info.depth - 1 if skip is None else skip
    pad = np.concatenate([np.full(w, 10, dtype=np.uint8), a])
    c = cls[pad].astype(np.int64)
    st = np.full(a.size, info.classes, dtype=np.int64)
    for j in range(w + 1):
        st = table[st + c[j:j + a.size]]
    return st


def count_lines(info, cls, table, a):
    succ = lane_states(info, cls, table, a) == 0
    line = np.concatenate([[0], np.cumsum(a == 10)[:-1]])
    return int(np.unique(line[succ & (a != 10)]).size)


def sequential_states(info, cls, table, a):
    st = info.classes
    out = np.empty(a.size, dtype=np.int64)
    for k, b in enumerate(a.tolist()):
        st = int(table[st + cls[b]])
        out[k] = st
    return out


def _targets():
    return [("golden", n) for n in G.pattern_names()] + [("config", os.path.basename(p)[:-5]) for p in CONFIGS]


def _path(kind, name):
    return G.pattern_path(name) if kind == "golden" else os.path.join(O.ROOT, "ugrep_b200", "patterns", name + ".ugxp")


@pytest.mark.parametrize("kind,name", _targets())
def test_search_automaton_counts_lines_as_the_oracle(kind, name):
    path = _path(kind, name)
    info, cls, table = describe(path)
    if not info.eligible:
        pytest.skip("refused: %d" % info.refusal)
    assert 1 <= info.depth <= 16 and info.states * info.classes <= 65536 and info.table_bytes <= 128 * 1024
    assert (table % info.classes == 0).all() and table.max() < info.states * info.classes
    assert (table[:info.classes] == 0).sum() == info.classes - 1  # MATCHED stays MATCHED except on '\n'
    assert table[cls[10]] == info.classes and table[info.classes + cls[10]] == info.classes
    op = O.OraclePattern(path)
    inputs = []
    if kind == "golden":
        inputs += [data for _, data in G.cases(name)]
    else:
        inputs += [corpus.block(c, 3 << 20).tobytes() for c in ("c2", "c2s", "c4")]
    for data in inputs:
        a = np.frombuffer(data, dtype=np.uint8)
        assert count_lines(info, cls, table, a) == op.count_lines(data)


def test_eligibility_of_the_configs():
    pat = os.path.join(O.ROOT, "ugrep_b200", "patterns")
    c2, _, _ = describe(os.path.join(pat, "c2.ugxp"))
    assert c2.eligible == 1 and c2.depth == 10
    assert c2.table_bytes <= 128 * 1024 and c2.states < 4507
    assert describe(os.path.join(pat, "c1.ugxp"))[0].refusal == ROUTE   # a literal's `one`: the literal kernel
    assert describe(os.path.join(pat, "c3.ugxp"))[0].refusal in (META, ROUTE)   # word boundaries; no proven cover
    assert describe(os.path.join(pat, "c5.ugxp"))[0].refusal in (META, CYCLE, DEPTH, ROUTE)   # look-back


def test_refusals_are_the_documented_ones():
    seen = set()
    for kind, name in _targets():
        info, _, _ = describe(_path(kind, name))
        assert info.eligible == (info.refusal == OK)
        assert info.refusal in (OK, META, ACC0, CYCLE, DEPTH, NEWLINE, SIZE, ROUTE)
        if info.refusal in (META, ACC0, CYCLE):
            assert info.states == 0 and info.table_bytes == 0
        seen.add(info.refusal)
    assert OK in seen and ROUTE in seen


def test_the_3000_word_list_is_refused_by_size(tmp_path):
    """tools/big_list.py's 3,000 words: their automaton outgrows the 128 KiB budget, so `-c` keeps
    count_lines_stream_kernel for them"""
    from ugrep_b200 import api
    opc, pf = api.compile_words(corpus.words_list(11, 3000))
    path = str(tmp_path / "w3000.ugxp")
    api.write_ugxp(path, opc, pf)
    info, _, _ = describe(path)
    assert info.refusal == SIZE and info.depth <= 16


def test_warm_up_gives_the_line_start_state():
    pat = os.path.join(O.ROOT, "ugrep_b200", "patterns")
    info, cls, table = describe(os.path.join(pat, "c2.ugxp"))
    a = corpus.block("c2", 200000)
    # the whole buffer from its start, one byte after the other (the first line starts at offset 0)
    seq = sequential_states(info, cls, table, a)
    rng = np.random.default_rng(5)
    for w in (info.depth - 1, 15):
        warm = lane_states(info, cls, table, a, skip=w)
        # where a pass from the line start is not MATCHED, the warm-up state is exactly its state; where it is MATCHED,
        # the warm-up pass may still hold the undecided set, but then the first success of the line is found by both
        assert ((seq == 0) | (warm == seq)).all()
        assert (warm == 0).sum() <= (seq == 0).sum() and ((warm == 0) <= (seq == 0)).all()
    for x in rng.integers(0, a.size - 64, 200):
        st = info.classes
        for b in a[x - min(x, info.depth - 1):x + 1].tolist():
            st = int(table[st + cls[b]])
        assert st == seq[x] or seq[x] == 0
