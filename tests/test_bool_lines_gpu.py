"""Boolean line queries on the GPU (ugx_count_lines_bool / ugx_find_lines_bool*, `--and` / `--andnot` / `--bool`, `-v`
included): every record byte for byte against the oracle's derivation (bool_oracle.py) and totals.matches against their
count, on golden pattern pairs with seeded random CNFs through every selection route, three-term queries on config
blocks with large bases, the equivalence with ugx_find_lines, edge inputs, host / pinned / device / misaligned buffers,
the limits and argument checks, overflow and paging, the match arena alongside, and the reference CLI where it
travelled."""
import ctypes as C
import os
import zlib

import numpy as np
import pytest

import bool_oracle as BO
import golden_lib as G
import lines_oracle as LO
import oracle_lib as O
from test_find_lines_gpu import EDGE
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu
PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")
ROUTES = {"default": {}, "no_span": {"no_span": 1}, "force_generic": {"force_generic": 1}}
FIXED = [[[0]], [[~0]], [[0], [1]], [[0], [~1]], [[0, 1]], [[~0, ~1]], [[0, ~0]], []]


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api as A
    return A


def cfg(name):
    return os.path.join(PAT_DIR, name + ".ugxp")


class Cached:
    """the oracle's line records of one buffer per pattern, polarity and bases, computed once"""

    def __init__(self, op, data):
        self.op, self.data, self.memo = op, data, {}

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        assert data is self.data
        key = (invert, base_offset, base_line)
        if key not in self.memo:
            self.memo[key] = self.op.find_lines(data, invert, base_offset, base_line)
        return self.memo[key]


class DeviceLines:
    """the derivation's input from the device's own find_lines (tested against the oracle in test_find_lines_gpu.py),
    for inputs too large for the CPU oracle"""

    def __init__(self, sc, pat):
        self.sc, self.pat = sc, pat

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        return self.sc.find_lines(self.pat, data, invert=invert, base_offset=base_offset, base_line=base_line)[0]


def random_cnfs(rng, k, count):
    out = []
    for _ in range(count):
        cnf = []
        for _ in range(int(rng.integers(1, 4))):
            lits = rng.choice(2 * k, size=int(rng.integers(1, 3)), replace=False)
            cnf.append([int(x) // 2 if x % 2 == 0 else ~(int(x) // 2) for x in lits])
        out.append(cnf)
    return out


def check(sc, pats, ops, data, cnf, invert, what, base_offset=0, base_line=0, count=True):
    rec, tot = sc.find_lines_bool(pats, cnf, data, invert, base_offset, base_line)
    want = BO.find_lines_bool(ops, cnf, data, invert, base_offset, base_line)
    assert len(rec) == len(want) == tot.matches, (what, cnf, invert, len(rec), len(want), tot)
    assert rec.tobytes() == want.tobytes(), (what, cnf, invert)
    assert tot.flags & 1 and tot.kernel == "bool_count_kernel", tot
    if count:
        cnt = sc.count_lines_bool(pats, cnf, data, invert)
        assert cnt.matches == len(want) and cnt.newlines == tot.newlines, (what, cnf, invert, cnt)
    return rec, tot


def load_pair(api, name):
    """the golden pattern `name` and the next golden pattern after it that the library takes"""
    try:
        a = api.Pattern.load(G.pattern_path(name), 0)
    except api.UgxError as ex:
        assert ex.code == 2, ex
        pytest.skip("out of scope: %s" % ex)
    names = G.pattern_names()
    i = names.index(name)
    for k in range(1, len(names)):
        other = names[(i + k) % len(names)]
        try:
            return a, api.Pattern.load(G.pattern_path(other), 0), other
        except api.UgxError as ex:
            assert ex.code == 2, ex
    raise AssertionError("no second pattern")


@pytest.mark.parametrize("name", G.pattern_names())
def test_golden_pairs_every_route(api, name):
    """every golden pattern with the next one: on each route, all the pattern's golden cases joined into one buffer (each
    case a run of lines) under the CNFs; on the default route also every case alone, which keeps each case's own end
    of buffer, under a seeded random CNF, the polarities alternating"""
    a, b, other = load_pair(api, name)
    oa, ob = LO.oracle(G.pattern_path(name)), LO.oracle(G.pattern_path(other))
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    cnfs = FIXED + random_cnfs(rng, 2, 3)
    cases = [data for _, data in G.cases(name)] + EDGE[:-1]
    joined = b"\n".join(cases)
    ops = [Cached(oa, joined), Cached(ob, joined)]
    for route, opts in ROUTES.items():
        sc = api.Scanner(0)
        for k, v in opts.items():
            sc.set_option(k, v)
        # the routes differ only in the terms' selection: the other routes take the two-term CNFs and the random ones
        for cnf in (cnfs if route == "default" else cnfs[2:6] + cnfs[8:]):
            for inv in (False, True):
                check(sc, [a, b], ops, joined, cnf, inv, (name, other, route), count=route == "default")
    sc = api.Scanner(0)
    for i, data in enumerate(cases):
        ops = [Cached(oa, data), Cached(ob, data)]
        check(sc, [a, b], ops, data, random_cnfs(rng, 2, 1)[0], i % 2 == 1, (name, other, data[:40]), count=i % 3 == 0)


def literal_term(api, tmp_path, text):
    """a library-compiled literal (Pattern.literal) and the oracle on the same words written out as UGXP"""
    opc, pf = api.compile_literal(text)
    path = str(tmp_path / ("lit_%s.ugxp" % text.hex()))
    api.write_ugxp(path, opc, pf)
    return api.Pattern.literal(text, 0), LO.oracle(path)


THREE = {"c2": ("c2", [b"the", b"and"]), "c3": ("c3", [b"ing", None]), "c4": ("c4", [b"the", b"a"]),
         "c5": ("c5", [b"ERROR", b"555"])}


@pytest.mark.parametrize("cname", list(THREE))
def test_config_blocks_three_terms(api, tmp_path, cname):
    """4 MiB blocks (hundreds of regions and line blocks), three terms of which two are library-compiled literals (c3:
    c3 and c3b, whose prefilter never fires / fires), an unterminated last line, offsets beyond 2^32, line numbers at
    2^40"""
    sc = api.Scanner(0)
    first, lits = THREE[cname]
    pats, ops = [api.Pattern.load(cfg(first), 0)], [LO.oracle(cfg(first))]
    for text in lits:
        if text is None:
            pats.append(api.Pattern.load(cfg("c3b"), 0))
            ops.append(LO.oracle(cfg("c3b")))
        else:
            p, o = literal_term(api, tmp_path, text)
            pats.append(p)
            ops.append(o)
    data = corpus.block(cname, 4 << 20)
    cut = data[:len(data) - 5]
    rng = np.random.default_rng(11)
    cnfs = [[[0], [1]], [[0], [~2]], [[1, 2], [~0]], [[0, 1, 2]], [[~1]]] + random_cnfs(rng, 3, 3)
    for buf in (data, cut):
        cached = [Cached(o, buf) for o in ops]
        for base_offset, base_line in ((0, 0), ((1 << 33) + 5, 1 << 40)):
            for cnf in cnfs:
                for inv in (False, True):
                    check(sc, pats, cached, buf, cnf, inv, cname, base_offset, base_line)


@pytest.mark.parametrize("name,cname", [("c1", "c1"), ("c2", "c2"), ("c3b", "c3"), ("c5", "c5"), ("w_the", "c1")])
def test_one_clause_equals_find_lines(api, name, cname):
    import torch
    sc = api.Scanner(0)
    path = cfg(name) if name != "w_the" else G.pattern_path(name)
    pat = api.Pattern.load(path, 0)
    dev = torch.from_numpy(corpus.block(cname, 2 << 20)).cuda()
    for inv in (False, True):
        lines, lt = sc.find_lines(pat, dev, invert=inv, base_offset=7, base_line=3)
        for cnf, negated in (([[0]], False), ([[~0]], True)):
            rec, tot = sc.find_lines_bool([pat], cnf, dev, inv != negated, 7, 3)
            assert tot.matches == len(rec) == len(lines) and tot.newlines == lt.newlines, (name, inv, cnf)
            for f in ("line", "bol", "eol"):
                assert np.array_equal(rec[f], lines[f]), (name, inv, cnf, f)
            assert (rec["cap"] == (0 if inv else 1)).all() and (rec["offset"] == rec["bol"]).all()
            assert not rec["len"].any()


def test_edge_inputs(api):
    """an empty buffer, only '\\n', no '\\n', lines of 80 KB across regions, and a 64 MiB line"""
    import torch
    sc = api.Scanner(0)
    c1, c5 = api.Pattern.load(G.pattern_path("c1"), 0), api.Pattern.load(cfg("c5"), 0)
    o1, o5 = LO.oracle(G.pattern_path("c1")), LO.oracle(cfg("c5"))
    H = b"Sherlock Holmes"
    rng = np.random.default_rng(5)
    words = np.array([b"x", b" ", b"ERROR", b"y "], dtype=object)
    long = [b"".join(rng.choice(words, 30000)) for _ in range(4)]
    cases = [b"", b"\n", b"\n" * 100000, b"ERROR " + H, (b"ERROR x " * 30000) + H,
             b"\n".join(s + H + s for s in long) + b"\n", b"\n".join(long) + b" WARN"]
    for data in cases:
        for cnf in ([[0], [~1]], [[0, 1]], [[~0], [~1]], []):
            for inv in (False, True):
                check(sc, [c1, c5], [Cached(o1, data), Cached(o5, data)], data, cnf, inv, data[:30])
    tot = sc.find_lines_bool([c1, c5], [], b"")[1]
    assert (tot.matches, tot.launches, tot.newlines) == (0, 0, 0)
    # a 64 MiB line between short ones: the derivation's input from the device's find_lines
    big = b"y" * (64 << 20)
    data = b"a ERROR\n" + big + H + big + b"\nERROR\n" + H
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    dl = [DeviceLines(sc, c1), DeviceLines(sc, c5)]
    for cnf in ([[0], [~1]], [[0, 1]]):
        for inv in (False, True):
            rec, _ = check(sc, [c1, c5], dl, dev, cnf, inv, cnf)
            if cnf == [[0], [~1]] and not inv:
                assert len(rec) == 2 and int(rec["eol"][0]) - int(rec["bol"][0]) == (128 << 20) + len(H)


def test_config3_never_fires_and_hand_over(api):
    sc = api.Scanner(0)
    c3, c5 = api.Pattern.load(cfg("c3"), 0), api.Pattern.load(cfg("c5"), 0)
    o3, o5 = LO.oracle(cfg("c3")), LO.oracle(cfg("c5"))
    data = corpus.block("c3", 1 << 20)
    for cnf in ([[0]], [[~0]], [[0, 1]], [[~0], [1]]):
        for inv in (False, True):
            check(sc, [c3, c5], [Cached(o3, data), Cached(o5, data)], data, cnf, inv, "c3")
    # c5's span selection hands this buffer over: the flag is set, the result still exact
    dot = api.Pattern.load(G.pattern_path("dotstar"), 0)
    od = LO.oracle(G.pattern_path("dotstar"))
    c1 = api.Pattern.load(G.pattern_path("c1"), 0)
    o1 = LO.oracle(G.pattern_path("c1"))
    for other, oo, data in ((c5, o5, b"x" * 100000 + b" ERROR 555-12"),
                            (dot, od, b"a" + b"q" * 70000 + b"b\n" + b"ab\n" * 5)):
        for cnf in ([[0]], [[~0], [1]], [[0, 1]]):
            for inv in (False, True):
                _, tot = check(sc, [other, c1], [Cached(oo, data), Cached(o1, data)], data, cnf, inv, "handover")
                assert tot.flags & 2, tot


def test_host_pinned_device_and_misaligned_buffers(api):
    import torch
    sc = api.Scanner(0)
    c2, c5 = api.Pattern.load(cfg("c2"), 0), api.Pattern.load(cfg("c5"), 0)
    o2, o5 = LO.oracle(cfg("c2")), LO.oracle(cfg("c5"))
    base = corpus.block("c5", 400000)
    dev = torch.from_numpy(base).cuda()
    for lo, hi in ((0, len(base)), (3, 300001), (17, 123457)):
        data = base[lo:hi]
        ops = [Cached(o5, data), Cached(o2, data)]
        for cnf, inv in (([[0], [~1]], False), ([[0, 1]], True)):
            want = BO.find_lines_bool(ops, cnf, data, inv, 1 << 40, 1 << 33)
            for src in (data, dev[lo:hi], torch.from_numpy(data.copy()).pin_memory().numpy()):
                rec, tot = sc.find_lines_bool([c5, c2], cnf, src, inv, 1 << 40, 1 << 33)
                assert rec.tobytes() == want.tobytes() and tot.matches == len(want), (lo, hi, cnf, inv)
                assert sc.count_lines_bool([c5, c2], cnf, src, inv).matches == len(want)


def raw_args(api, sc, pats, clauses, data):
    arr = (C.c_void_p * max(1, len(pats)))(*[p._h if p is not None else None for p in pats])
    return (sc._h, arr, len(pats), clauses, len(clauses) if clauses is not None else 0, C.c_void_p(data.ctypes.data),
            len(data))


def test_limits_and_argument_checks(api):
    sc = api.Scanner(0)
    L = api.lib()
    c1 = api.Pattern.load(G.pattern_path("c1"), 0)
    o1 = LO.oracle(G.pattern_path("c1"))
    data = corpus.block("c1", 300000)
    # 32 patterns pass (the same pattern 32 times: every bit of a matching line's mask is set)
    rec, tot = sc.find_lines_bool([c1] * 32, [[31], [~0, 5]], data)
    want = o1.find_lines(data)
    assert np.array_equal(rec["line"], want["line"]) and (rec["cap"] == 0xffffffff).all()
    assert tot.launches >= 32
    t = api._Totals()
    cnt, dev = C.c_uint64(), C.c_void_p()
    out = np.zeros(16, dtype=api.LINE_DTYPE)
    one = api.bool_clauses([[0]])

    def count(pats, clauses, flags=0, buf=data, n=None):
        a = list(raw_args(api, sc, pats, clauses, buf))
        if n is not None:
            a[6] = n
        return L.ugx_count_lines_bool(*a, flags, C.byref(t))

    def find(pats, clauses, flags=0):
        return L.ugx_find_lines_bool(*raw_args(api, sc, pats, clauses, data), 0, 0, flags, out.ctypes.data, 16,
                                     C.byref(cnt), C.byref(t))

    def find_dev(pats, clauses, flags=0):
        return L.ugx_find_lines_bool_device(*raw_args(api, sc, pats, clauses, data), 0, 0, flags, C.byref(dev),
                                            C.byref(cnt), C.byref(t))

    assert count([c1] * 33, one) == 2 and find([c1] * 33, one) == 2 and find_dev([c1] * 33, one) == 2
    many = api.bool_clauses([[0]] * 65)
    assert count([c1], many) == 2 and find([c1], many) == 2 and find_dev([c1], many) == 2
    assert count([c1], api.bool_clauses([[0]] * 64)) == 0 and t.matches == len(want)
    empty = (api.BoolClause * 1)()
    for call in (count, find, find_dev):
        assert call([c1], empty) == 1                               # an empty clause
        assert call([c1], api.bool_clauses([[1]])) == 1             # a bit at or above npatterns
        assert call([c1], api.bool_clauses([[~1]])) == 1
        assert call([c1, c1], api.bool_clauses([[0], [~2]])) == 1
        assert call([], one) == 1                                   # npatterns == 0
        assert call([c1, None], one) == 1                           # a null pattern
        assert call([c1], one, 2) == 1 and call([c1], one, 3) == 1  # flags
        assert call([c1], None) == (5 if call is find else 0)       # no clauses: every line (overflows out[16])
    assert count([c1], None) == 0 and t.matches == len(o1.find_lines(data)) + len(o1.find_lines(data, True))
    # a null clause array with nclauses > 0, a null pattern array, a null scanner, a null buffer with nbytes > 0
    a = list(raw_args(api, sc, [c1], one, data))
    assert L.ugx_count_lines_bool(a[0], a[1], 1, None, 1, a[5], a[6], 0, C.byref(t)) == 1
    assert L.ugx_count_lines_bool(a[0], None, 1, one, 1, a[5], a[6], 0, C.byref(t)) == 1
    assert L.ugx_count_lines_bool(None, a[1], 1, one, 1, a[5], a[6], 0, C.byref(t)) == 1
    assert L.ugx_count_lines_bool(a[0], a[1], 1, one, 1, None, 5, 0, C.byref(t)) == 1
    assert L.ugx_count_lines_bool(a[0], a[1], 1, one, 1, None, 0, 0, C.byref(t)) == 0 and t.matches == 0
    assert L.ugx_find_lines_bool(a[0], a[1], 1, one, 1, a[5], a[6], 0, 0, 0, None, 0, C.byref(cnt), C.byref(t)) == 5
    assert L.ugx_find_lines_bool(a[0], a[1], 1, one, 1, a[5], a[6], 0, 0, 0, None, cnt.value, C.byref(cnt),
                                 C.byref(t)) == 1
    # a pattern on another device, where there is one
    import torch
    if torch.cuda.device_count() > 1:
        other = api.Pattern.load(G.pattern_path("c1"), 1)
        assert count([c1, other], one) == 1


def test_overflow_paging_and_the_match_arena(api):
    sc = api.Scanner(0)
    L = api.lib()
    c5, c2 = api.Pattern.load(cfg("c5"), 0), api.Pattern.load(cfg("c2"), 0)
    o5, o2 = LO.oracle(cfg("c5")), LO.oracle(cfg("c2"))
    data = corpus.block("c5", 1 << 20)
    other = corpus.block("c2", 1 << 20)
    ops = [Cached(o5, data), Cached(o2, data)]
    want = BO.find_lines_bool(ops, [[0], [~1]], data, False, 1 << 33, 9)
    assert len(want) > 100
    tm = sc.find_all_device(c2, other)
    clauses = api.bool_clauses([[0], [~1]])
    pats = (C.c_void_p * 2)(c5._h, c2._h)
    out = np.zeros(len(want), dtype=api.LINE_DTYPE)
    cnt, t = C.c_uint64(), api._Totals()
    args = (sc._h, pats, 2, clauses, 1 + 1, C.c_void_p(data.ctypes.data), len(data), 1 << 33, 9, 0)
    assert L.ugx_find_lines_bool(*args, out.ctypes.data, len(want) - 1, C.byref(cnt), C.byref(t)) == 5
    assert cnt.value == len(want) == t.matches
    paged = np.concatenate([sc.fetch_lines(i, min(97, len(want) - i)) for i in range(0, len(want), 97)])
    assert paged.tobytes() == want.tobytes()
    with pytest.raises(api.UgxError):
        sc.fetch_lines(len(want), 1)
    assert L.ugx_find_lines_bool(*args, out.ctypes.data, len(want), C.byref(cnt), C.byref(t)) == 0
    assert out.tobytes() == want.tobytes()
    # the find_all_device result is still fetchable after the Boolean calls
    assert sc.fetch(0, tm.matches).tobytes() == o2.find_all(other).tobytes()
    # ugx_count_lines_bool leaves the line arena at zero records
    assert sc.count_lines_bool([c5, c2], [[0], [~1]], data).matches == len(want)
    with pytest.raises(api.UgxError):
        sc.fetch_lines(0, 1)
    assert sc.fetch(0, tm.matches).tobytes() == o2.find_all(other).tobytes()


REF_QUERIES = [
    ("c5", [b"ERROR", b"555"], ["-e", "ERROR", "--and", "-e", "555"], [[0], [1]]),
    ("c5", [b"ERROR", b"555"], ["ERROR", "--andnot", "555"], [[0], [~1]]),
    ("c5", [b"ERROR", b"WARN", b"555"], ["--bool", "ERROR|WARN -555"], [[0, 1], [~2]]),
    ("c1", [b"Sherlock", b"Holmes", b"Watson"], ["--bool", "Sherlock Holmes|Watson"], [[0], [1, 2]]),
]


@pytest.mark.skipif(not O.have_reference(), reason="oracle/_ref (the built reference) did not travel")
@pytest.mark.parametrize("q", range(len(REF_QUERIES)))
def test_against_the_reference_cli(api, q):
    """`ugrep -F -c` and `ugrep -F -n` with --and / --andnot / --bool against the library's count and records"""
    cname, words, cli, cnf = REF_QUERIES[q]
    sc = api.Scanner(0)
    pats = [api.Pattern.literal(w, 0) for w in words]
    data = corpus.block(cname, 2 << 20)
    rc, ref = O.ref_cli(["-F", "-c", *cli], data)
    assert ref == b"%d\n" % sc.count_lines_bool(pats, cnf, data).matches, (cli, ref)
    rec, _ = sc.find_lines_bool(pats, cnf, data)
    raw = data.tobytes()
    mine = b"".join(b"%d:%s\n" % (int(r["line"]), raw[int(r["bol"]):int(r["eol"])]) for r in rec)
    rc, ref = O.ref_cli(["-F", "-n", *cli], data)
    assert mine == ref, cli
