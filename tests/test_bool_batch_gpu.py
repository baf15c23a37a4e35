"""Boolean line queries over many files on the GPU (ugx_count_lines_bool_batch / ugx_find_lines_bool_batch, `ugrep -r
--and` / `--andnot` / `--bool`, `-c`, `-l`, `-v`): every file's slice rec[first[i]:first[i + 1]] byte for byte against
the oracle's per-file derivation (test_bool_batch.find_lines_bool_batch), or against ugx_find_lines_bool /
ugx_count_lines_bool on each file alone where the inputs are too large for the CPU oracle, in both polarities, with
counts and first[].  Covers golden pattern pairs, three-term queries on config blocks cut into files, the padding
between files, line blocks spanning many files and files spanning many line blocks, empty files everywhere, a source
tree's worth of files, host / pinned / device buffers, the equivalence with ugx_find_lines_batch, the limits and
argument checks, overflow and paging, the two record arenas, and the reference CLI where it travelled."""
import ctypes as C
import os
import subprocess
import tempfile
import zlib

import numpy as np
import pytest

import golden_lib as G
import lines_oracle as LO
import oracle_lib as O
from test_batch_gpu import make_files
from test_batch_records_gpu import pack
from test_bool_batch import find_lines_bool_batch
from test_bool_lines_gpu import FIXED, load_pair, random_cnfs
from test_find_lines_gpu import EDGE
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu
PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")
H = b"Sherlock Holmes"


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api as A
    return A


def cfg(name):
    return os.path.join(PAT_DIR, name + ".ugxp")


class Memo:
    """an oracle's line records per (file, polarity), computed once"""

    def __init__(self, op):
        self.op, self.memo = op, {}

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        key = (bytes(data), invert, base_offset, base_line)
        if key not in self.memo:
            self.memo[key] = self.op.find_lines(data, invert, base_offset, base_line)
        return self.memo[key]


class DeviceLines:
    """the derivation's input from the device's own ugx_find_lines, for inputs too large for the CPU oracle"""

    def __init__(self, sc, pat):
        self.sc, self.pat = sc, pat

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        return self.sc.find_lines(self.pat, data, invert=invert, base_offset=base_offset, base_line=base_line)[0]


def line_count(f):
    return f.count(b"\n") + (1 if len(f) and not f.endswith(b"\n") else 0)


def check(sc, pats, ops, files, cnf, invert, what, src=None, count=True):
    """both forms of the batch against the derivation; `src` is the packed input when not the list itself"""
    src = files if src is None else src
    rec, first, tot = sc.find_lines_bool_batch(pats, cnf, src, invert)
    want, wfirst, wcounts = find_lines_bool_batch(ops, cnf, files, invert)
    assert len(rec) == len(want) == tot.matches, (what, cnf, invert, len(rec), len(want), tot)
    assert np.array_equal(first, wfirst), (what, cnf, invert)
    if rec.tobytes() != want.tobytes():
        for i in range(len(files)):
            a, b = rec[int(first[i]):int(first[i + 1])], want[int(wfirst[i]):int(wfirst[i + 1])]
            assert a.tobytes() == b.tobytes(), (what, cnf, invert, "file", i, files[i][:40], a[:4], b[:4])
        raise AssertionError((what, cnf, invert))
    assert tot.newlines == sum(f.count(b"\n") for f in files), (what, tot)
    assert tot.flags & 1 and tot.kernel == "bool_count_kernel", tot
    if count:
        counts, ct = sc.count_lines_bool_batch(pats, cnf, src, invert)
        assert np.array_equal(counts, wcounts) and ct.matches == len(want), (what, cnf, invert)
        assert ct.newlines == tot.newlines and ct.kernel == "bool_count_kernel", ct
    return rec, first, tot


@pytest.mark.parametrize("name", G.pattern_names())
def test_golden_pairs(api, name):
    """every golden pattern with the next one the library takes: the pattern's golden cases plus the edge inputs as
    files, under the fixed CNFs and seeded random ones, both polarities"""
    a, b, other = load_pair(api, name)
    ops = [Memo(LO.oracle(G.pattern_path(name))), Memo(LO.oracle(G.pattern_path(other)))]
    rng = np.random.default_rng(zlib.crc32(name.encode()) + 1)
    files = [data for _, data in G.cases(name)] + EDGE
    sc = api.Scanner(0)
    for k, cnf in enumerate(FIXED + random_cnfs(rng, 2, 3)):
        for inv in (False, True):
            check(sc, [a, b], ops, files, cnf, inv, (name, other), count=k % 2 == 0 or inv)


THREE = {"c5": [b"ERROR", b"555"], "c2": [b"the", b"and"], "c4": [b"the", b"a"]}


def literal_term(api, tmp_path, text):
    opc, pf = api.compile_literal(text)
    path = str(tmp_path / ("lit_%s.ugxp" % text.hex()))
    api.write_ugxp(path, opc, pf)
    return api.Pattern.literal(text, 0), LO.oracle(path)


def three_terms(api, tmp_path, cname):
    pats, ops = [api.Pattern.load(cfg(cname), 0)], [Memo(LO.oracle(cfg(cname)))]
    for text in THREE[cname]:
        p, o = literal_term(api, tmp_path, text)
        pats.append(p)
        ops.append(Memo(o))
    return pats, ops


@pytest.mark.parametrize("cname", list(THREE))
def test_config_blocks_cut_into_files(api, tmp_path, cname):
    """make_files: unterminated last lines, files of 16383 / 16384 / 16385 bytes, 70 000-byte files across tiles; three
    terms of which two are library-compiled literals"""
    sc = api.Scanner(0)
    pats, ops = three_terms(api, tmp_path, cname)
    files = make_files(cname, np.random.default_rng(21), 40)
    rng = np.random.default_rng(12)
    for cnf in [[[0], [1]], [[0], [~2]], [[1, 2], [~0]], [[0, 1, 2]], [[~1]]] + random_cnfs(rng, 3, 2):
        for inv in (False, True):
            check(sc, pats, ops, files, cnf, inv, cname)


def test_padding_is_never_text(api, tmp_path):
    """the same files packed with 'X' padding and with padding full of '\\n' and of the terms' text"""
    sc = api.Scanner(0)
    pats, ops = three_terms(api, tmp_path, "c5")
    files = make_files("c5", np.random.default_rng(4), 30) + [b"ERROR 555", b"", b"x"]
    for cnf in ([[0], [1]], [[0, ~2]], []):
        for inv in (False, True):
            rec, first, _ = check(sc, pats, ops, files, cnf, inv, "X", src=pack(files, b"X"))
            for pad in (b"\n", b"ERROR 555\n\n", b"the\nand ERROR\n555"):
                r2, f2, t2 = sc.find_lines_bool_batch(pats, cnf, pack(files, pad), inv)
                assert r2.tobytes() == rec.tobytes() and np.array_equal(f2, first), (pad, cnf, inv)
                assert t2.newlines == sum(f.count(b"\n") for f in files)
                c2, _ = sc.count_lines_bool_batch(pats, cnf, pack(files, pad), inv)
                assert np.array_equal(c2, np.diff(first.astype(np.int64)).astype(np.uint64)), (pad, cnf, inv)


def test_line_block_boundaries(api):
    """thousands of few-line files (one 8192-line block spans many files), a file of more than 8192 lines, a line of
    more than 1 MiB, and empty files and files that are only '\\n' interleaved everywhere, first and last included"""
    sc = api.Scanner(0)
    c1, c5 = api.Pattern.load(G.pattern_path("c1"), 0), api.Pattern.load(cfg("c5"), 0)
    ops = [Memo(LO.oracle(G.pattern_path("c1"))), Memo(LO.oracle(cfg("c5")))]
    base = corpus.block("c5", 1 << 20).tobytes()
    lines = base.split(b"\n")
    rng = np.random.default_rng(31)
    few = []
    at = 0
    for k in range(6000):
        n = int(rng.integers(1, 5))
        f = b"\n".join(lines[at:at + n]) + (b"\n" if k % 3 else b"")
        if k % 7 == 0:
            f += b" " + H
        few.append(f)
        at = (at + n) % (len(lines) - 8)
    many = b"\n".join(lines[:9000]) + b"\n" + H
    assert line_count(many) > 8192
    long = b"ERROR " + b"y" * (1 << 20) + H + b" z\nshort ERROR\n" + b"q" * (1 << 20)
    blanks = [b"", b"\n", b"", b"\n"]
    files = blanks + few[:3000] + blanks + [many] + blanks + [long] + few[3000:] + blanks
    assert sum(line_count(f) for f in files) > 3 * 8192
    for cnf in ([[0], [~1]], [[0, 1]], [[~0], [~1]], []):
        for inv in (False, True):
            check(sc, [c1, c5], ops, files, cnf, inv, ("blocks", cnf))
    for inv in (False, True):
        rec, first, _ = sc.find_lines_bool_batch([c1, c5], [[0, 1]], files, inv)
        for i in range(len(blanks)):
            assert first[i] == first[i + 1] or (files[i] == b"\n" and first[i + 1] - first[i] == int(inv))


def test_a_source_tree_worth_of_files(api, tmp_path):
    """20 000 files of U(0, 4 KiB): a sample of files against ugx_find_lines_bool / ugx_count_lines_bool on each file
    alone, and the counts against first[]"""
    sc = api.Scanner(0)
    pats, _ = three_terms(api, tmp_path, "c5")
    base = corpus.block("c5", 2 << 20).tobytes()
    rng = np.random.default_rng(8)
    files = []
    for _ in range(20000):
        lo = int(rng.integers(0, len(base) - 4096))
        files.append(base[lo:lo + int(rng.integers(0, 4096))])
    sample = rng.integers(0, len(files), size=150)
    for cnf in ([[0], [~1]], [[1, 2]]):
        for inv in (False, True):
            rec, first, tot = sc.find_lines_bool_batch(pats, cnf, files, inv)
            counts, ct = sc.count_lines_bool_batch(pats, cnf, files, inv)
            assert np.array_equal(counts, np.diff(first.astype(np.int64)).astype(np.uint64)) and ct.matches == len(rec)
            assert tot.newlines == sum(f.count(b"\n") for f in files) and tot.matches == len(rec)
            for i in sample:
                want, wt = sc.find_lines_bool(pats, cnf, files[i], inv)
                assert rec[int(first[i]):int(first[i + 1])].tobytes() == want.tobytes(), (cnf, inv, i)
                assert int(counts[i]) == sc.count_lines_bool(pats, cnf, files[i], inv).matches


def test_host_pinned_and_device_buffers(api):
    import torch
    sc = api.Scanner(0)
    c2, c5 = api.Pattern.load(cfg("c2"), 0), api.Pattern.load(cfg("c5"), 0)
    ops = [Memo(LO.oracle(cfg("c5"))), Memo(LO.oracle(cfg("c2")))]
    files = make_files("c5", np.random.default_rng(6), 25)
    buf, begins, lens = pack(files)
    pinned = torch.from_numpy(buf.copy()).pin_memory()
    dev = torch.from_numpy(buf).cuda()
    for cnf, inv in (([[0], [~1]], False), ([[0, 1]], True), ([[~0]], False)):
        want, wfirst, wcounts = find_lines_bool_batch(ops, cnf, files, inv)
        for src in (buf, pinned.numpy(), dev):
            rec, first, tot = sc.find_lines_bool_batch([c5, c2], cnf, (src, begins, lens), inv)
            assert rec.tobytes() == want.tobytes() and np.array_equal(first, wfirst), (cnf, inv, type(src))
            counts, _ = sc.count_lines_bool_batch([c5, c2], cnf, (src, begins, lens), inv)
            assert np.array_equal(counts, wcounts), (cnf, inv)


@pytest.mark.parametrize("name,cname", [("c1", "c1"), ("c2", "c2"), ("c3b", "c3"), ("c3", "c3"), ("c5", "c5")])
def test_one_term_equals_find_lines_batch(api, name, cname):
    """K = 1: [[0]] gives ugx_find_lines_batch's records and [[~0]] its -v records, in line / bol / eol"""
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg(name), 0)
    files = make_files(cname, np.random.default_rng(9), 40)
    for inv in (False, True):
        lines, lfirst, lt = sc.find_lines_batch(pat, files, inv)
        for cnf, negated in (([[0]], False), ([[~0]], True)):
            rec, first, tot = sc.find_lines_bool_batch([pat], cnf, files, inv != negated)
            assert tot.matches == len(rec) == len(lines) and tot.newlines == lt.newlines, (name, inv, cnf)
            assert np.array_equal(first, lfirst), (name, inv, cnf)
            for f in ("line", "bol", "eol"):
                assert np.array_equal(rec[f], lines[f]), (name, inv, cnf, f)
            assert (rec["cap"] == (0 if inv else 1)).all() and (rec["offset"] == rec["bol"]).all()
            assert not rec["len"].any()


def raw_args(sc, pats, clauses, buf, begins, lens, nfiles=None):
    arr = (C.c_void_p * max(1, len(pats)))(*[p._h if p is not None else None for p in pats])
    return [sc._h, arr, len(pats), clauses, len(clauses) if clauses is not None else 0, C.c_void_p(buf.ctypes.data),
            buf.size, begins.ctypes.data if begins is not None else None,
            lens.ctypes.data if lens is not None else None, len(lens) if nfiles is None else nfiles]


def test_limits_and_argument_checks(api):
    """32 patterns and 64 clauses pass, 33 and 65 do not; every argument check fails before any device work, leaving
    the line arena and the match arena as they were"""
    sc = api.Scanner(0)
    L = api.lib()
    c1, c2 = api.Pattern.load(G.pattern_path("c1"), 0), api.Pattern.load(cfg("c2"), 0)
    o1 = LO.oracle(G.pattern_path("c1"))
    files = make_files("c1", np.random.default_rng(2), 12)
    buf, begins, lens = pack(files)
    rec, first, tot = sc.find_lines_bool_batch([c1] * 32, [[31], [~0, 5]], files)
    want = np.concatenate([o1.find_lines(f) for f in files])
    assert np.array_equal(rec["line"], want["line"]) and (rec["cap"] == 0xffffffff).all()
    assert tot.launches >= 32
    rec, _, _ = sc.find_lines_bool_batch([c1], [[0]] * 64, files)
    assert len(rec) == len(want)
    # the arenas the failing calls must leave alone
    other = corpus.block("c2", 300000)
    tm = sc.find_all_device(c2, other)
    lines_before = sc.find_lines_bool_batch([c1, c2], [[0, 1]], files)[0]
    matches_before = sc.fetch(0, tm.matches)
    assert len(lines_before) > 0 and tm.matches > 0
    t = api._Totals()
    cnt = C.c_uint64()
    fst = np.zeros(len(files) + 1, dtype=np.uint64)
    counts = np.zeros(len(files), dtype=np.uint64)
    out = np.zeros(16, dtype=api.LINE_DTYPE)
    one = api.bool_clauses([[0]])

    def count(a, flags=0, counts_ptr=counts.ctypes.data):
        return L.ugx_count_lines_bool_batch(*a, flags, counts_ptr, C.byref(t))

    def find(a, flags=0, first_ptr=fst.ctypes.data):
        return L.ugx_find_lines_bool_batch(*a, flags, first_ptr, out.ctypes.data, 16, C.byref(cnt), C.byref(t))

    def args(pats=(c1,), clauses=one, b=buf, bg=begins, ln=lens):
        return raw_args(sc, list(pats), clauses, b, bg, ln, len(files))

    empty = (api.BoolClause * 1)()
    misaligned = begins.copy()
    misaligned[1] += 8
    too_long = lens.copy()
    too_long[-1] = buf.size
    bad = [(2, args(pats=[c1] * 33)), (2, args(clauses=api.bool_clauses([[0]] * 65))),
           (1, args(clauses=empty)), (1, args(clauses=api.bool_clauses([[1]]))),
           (1, args(pats=[c1, c1], clauses=api.bool_clauses([[0], [~2]]))), (1, args(pats=[])),
           (1, args(pats=[c1, None])), (1, args(bg=misaligned)), (1, args(ln=too_long)),
           (1, args(bg=None)), (1, args(ln=None))]
    for k, (code, a) in enumerate(bad):
        assert count(a) == code and find(a) == code, k
    a = args()
    assert count(a, 2) == 1 and find(a, 3) == 1                        # flags
    assert count(a, 0, None) == 1 and find(a, 0, None) == 1            # a null counts / first
    n = list(a)
    n[3], n[4] = None, 1                                               # a null clause array with nclauses > 0
    assert count(n) == 1 and find(n) == 1
    n = list(a)
    n[0] = None                                                        # a null scanner
    assert count(n) == 1 and find(n) == 1
    n = list(a)
    n[5] = None                                                        # a null buffer with nbytes > 0
    assert count(n) == 1 and find(n) == 1
    assert sc.fetch_lines(0, len(lines_before)).tobytes() == lines_before.tobytes()
    with pytest.raises(api.UgxError):
        sc.fetch_lines(len(lines_before), 1)
    assert sc.fetch(0, tm.matches).tobytes() == matches_before.tobytes()
    import torch
    if torch.cuda.device_count() > 1:
        far = api.Pattern.load(G.pattern_path("c1"), 1)
        assert count(args(pats=[c1, far])) == 1


def test_overflow_paging_and_the_arenas(api, tmp_path):
    sc = api.Scanner(0)
    L = api.lib()
    pats, ops = three_terms(api, tmp_path, "c5")
    files = make_files("c5", np.random.default_rng(14), 30)
    want, wfirst, _ = find_lines_bool_batch(ops, [[0], [~1]], files)
    assert len(want) > 100
    other = corpus.block("c2", 1 << 20)
    c2 = api.Pattern.load(cfg("c2"), 0)
    tm = sc.find_all_device(c2, other)
    matches = sc.fetch(0, tm.matches)
    buf, begins, lens = pack(files)
    arr = (C.c_void_p * 3)(*[p._h for p in pats])
    clauses = api.bool_clauses([[0], [~1]])
    a = (sc._h, arr, 3, clauses, 2, C.c_void_p(buf.ctypes.data), buf.size, begins.ctypes.data, lens.ctypes.data,
         len(files), 0)
    out = np.zeros(len(want), dtype=api.LINE_DTYPE)
    fst = np.zeros(len(files) + 1, dtype=np.uint64)
    cnt, t = C.c_uint64(), api._Totals()
    assert L.ugx_find_lines_bool_batch(*a, fst.ctypes.data, out.ctypes.data, len(want) - 1, C.byref(cnt),
                                       C.byref(t)) == 5
    assert cnt.value == len(want) == t.matches and np.array_equal(fst, wfirst)
    paged = np.concatenate([sc.fetch_lines(i, min(97, len(want) - i)) for i in range(0, len(want), 97)])
    assert paged.tobytes() == want.tobytes()
    with pytest.raises(api.UgxError):
        sc.fetch_lines(len(want), 1)
    fst[:] = 0
    assert L.ugx_find_lines_bool_batch(*a, fst.ctypes.data, out.ctypes.data, len(want), C.byref(cnt),
                                       C.byref(t)) == 0
    assert out.tobytes() == want.tobytes() and np.array_equal(fst, wfirst)
    # out == NULL with cap == 0: the records stay on the device
    fst[:] = 0
    assert L.ugx_find_lines_bool_batch(*a, fst.ctypes.data, None, 0, C.byref(cnt), C.byref(t)) == 0
    assert cnt.value == len(want) and np.array_equal(fst, wfirst)
    assert sc.fetch_lines(0, len(want)).tobytes() == want.tobytes()
    # the match arena is untouched; the count form leaves zero line records
    assert sc.fetch(0, tm.matches).tobytes() == matches.tobytes()
    counts, ct = sc.count_lines_bool_batch(pats, [[0], [~1]], files)
    assert ct.matches == len(want) and np.array_equal(counts, np.diff(wfirst.astype(np.int64)).astype(np.uint64))
    with pytest.raises(api.UgxError):
        sc.fetch_lines(0, 1)
    assert sc.fetch(0, tm.matches).tobytes() == matches.tobytes()


def test_no_files_and_only_empty_files(api):
    sc = api.Scanner(0)
    c1, c5 = api.Pattern.load(G.pattern_path("c1"), 0), api.Pattern.load(cfg("c5"), 0)
    for inv in (False, True):
        rec, first, tot = sc.find_lines_bool_batch([c1, c5], [[0, 1]], [], inv)
        assert len(rec) == 0 and list(first) == [0] and tot.matches == 0 and tot.launches == 0
        counts, ct = sc.count_lines_bool_batch([c1, c5], [[0, 1]], [], inv)
        assert len(counts) == 0 and ct.matches == 0 and ct.launches == 0
        rec, first, tot = sc.find_lines_bool_batch([c1, c5], [], [b""] * 5, inv)
        assert len(rec) == 0 and list(first) == [0] * 6 and (tot.matches, tot.launches, tot.newlines) == (0, 0, 0)
        assert tot.kernel == "bool_count_kernel"
        counts, ct = sc.count_lines_bool_batch([c1, c5], [], [b""] * 5, inv)
        assert list(counts) == [0] * 5 and (ct.matches, ct.launches) == (0, 0)


REF_WORDS = [b"ERROR", b"555"]


@pytest.mark.skipif(not O.have_reference(), reason="oracle/_ref (the built reference) did not travel")
def test_against_the_reference_cli_over_a_tree(api):
    """`ugrep -F -rn -e ERROR --and -e 555 dir` and `ugrep -F -rc` against the batch's records and counts"""
    sc = api.Scanner(0)
    pats = [api.Pattern.literal(w, 0) for w in REF_WORDS]
    files = make_files("c5", np.random.default_rng(17), 12)[1:]
    names = ["f%03d.txt" % i for i in range(len(files))]
    rec, first, _ = sc.find_lines_bool_batch(pats, [[0], [1]], files)
    counts, _ = sc.count_lines_bool_batch(pats, [[0], [1]], files)
    with tempfile.TemporaryDirectory() as d:
        for name, f in zip(names, files):
            with open(os.path.join(d, name), "wb") as fh:
                fh.write(f)
        cli = [O.REF_UGREP, "--no-config", "-F", "-r", "--sort=name", "-e", "ERROR", "--and", "-e", "555"]
        got = subprocess.run(cli + ["-n", d], capture_output=True).stdout
        mine = b""
        for i, (name, f) in enumerate(zip(names, files)):
            for r in rec[int(first[i]):int(first[i + 1])]:
                mine += b"%s:%d:%s\n" % (os.path.join(d, name).encode(), int(r["line"]), f[int(r["bol"]):int(r["eol"])])
        assert sorted(got.splitlines()) == sorted(mine.splitlines())
        got = subprocess.run(cli + ["-c", d], capture_output=True).stdout
        ref = {}
        for line in got.splitlines():
            path, _, c = line.rpartition(b":")
            ref[os.path.basename(path).decode()] = int(c)
        for name, c in zip(names, counts):
            assert ref.get(name, 0) == int(c), name
