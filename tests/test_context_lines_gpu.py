"""Context lines on the GPU (ugx_find_context*, `ugrep -n -A/-B/-C`, `-v` included): every record byte for byte against
the oracle's derivation (context_oracle.py) on every selection route, the window arithmetic at large bases, lines of
64 MiB as context and as the selected line, config 3, host / pinned / device / misaligned buffers, overflow and paging,
the two record arenas side by side, the argument checks, and the batch form against the single-buffer form."""
import ctypes as C
import os

import numpy as np
import pytest

import context_oracle as CO
import golden_lib as G
import lines_oracle as LO
import oracle_lib as O
from test_batch_gpu import make_files
from test_batch_records_gpu import pack
from test_find_lines_gpu import EDGE
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu
PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")
ROUTES = {"default": {}, "no_span": {"no_span": 1}, "generic": {"force_generic": 1}}
M = CO.UINT32_MAX
WINDOWS = [(0, 0), (1, 0), (0, 1), (2, 2), (3, 7), (M, M)]


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api as A
    return A


def cfg(name):
    return os.path.join(PAT_DIR, name + ".ugxp")


class DeviceLines:
    """the derivation's input taken from the device's own find_lines (tested against the oracle in
    test_find_lines_gpu.py), for inputs too large for the CPU oracle"""

    def __init__(self, sc, pat):
        self.sc, self.pat = sc, pat

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        return self.sc.find_lines(self.pat, data, invert=invert, base_offset=base_offset, base_line=base_line)[0]


class Cached:
    """the oracle's line records of one buffer, computed once per polarity and bases"""

    def __init__(self, op, data):
        self.op, self.data, self.memo = op, data, {}

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        assert data is self.data
        key = (invert, base_offset, base_line)
        if key not in self.memo:
            self.memo[key] = self.op.find_lines(data, invert, base_offset, base_line)
        return self.memo[key]


def check(sc, pat, op, data, before, after, invert, what, base_offset=0, base_line=0):
    rec, tot = sc.find_context(pat, data, before, after, invert=invert, base_offset=base_offset, base_line=base_line)
    want = CO.find_context(op, data, before, after, invert, base_offset, base_line)
    assert len(rec) == len(want), (what, before, after, invert, len(rec), len(want))
    assert rec.tobytes() == want.tobytes(), (what, before, after, invert)
    assert tot.matches == int(CO.is_selected(want, invert).sum()), (what, tot)
    assert tot.flags & 1
    return rec, tot


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("name", G.pattern_names())
def test_golden_patterns_every_route(api, name, route):
    sc = api.Scanner(0)
    for k, v in ROUTES[route].items():
        sc.set_option(k, v)
    try:
        pat = api.Pattern.load(G.pattern_path(name), 0)
    except api.UgxError as ex:
        assert ex.code == 2, ex
        pytest.skip("out of scope: %s" % ex)
    op = LO.oracle(G.pattern_path(name))
    # EDGE's last input (two lines of 70 KB) is left to the config tests: on the general route every call reruns the
    # line-at-a-time selection over it
    for data in [data for _, data in G.cases(name)] + EDGE[:-1]:
        for inv in (False, True):
            lines = sc.find_lines(pat, data, invert=inv)[1]
            od = Cached(op, data)
            for b, a in WINDOWS:
                rec, tot = check(sc, pat, od, data, b, a, inv, (name, route, data[:40]))
                assert (tot.kernel, tot.flags, tot.newlines) == (lines.kernel, lines.flags, lines.newlines)
                if len(data) and tot.matches:
                    assert tot.launches >= lines.launches + 3 + (1 if inv else 0), tot
                if (b, a) == (0, 0):
                    assert rec.tobytes() == sc.find_lines(pat, data, invert=inv)[0].tobytes()


@pytest.mark.parametrize("name,cname", [("c1", "c1"), ("c2", "c2"), ("c3b", "c3"), ("c4", "c4"), ("c5", "c5")])
def test_config_blocks_with_large_bases(api, name, cname):
    """4 MiB blocks (hundreds of tiles and regions: windows reach across them), offsets beyond 2^32, line numbers near
    2^64 - 2^33 (the window arithmetic saturates instead of wrapping)"""
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg(name), 0)
    op = LO.oracle(cfg(name))
    data = corpus.block(cname, 4 << 20)
    cut = data[:len(data) - 5]  # unterminated last line
    od, oc = Cached(op, data), Cached(op, cut)
    for base_offset, base_line in ((0, 0), ((1 << 33) + 5, (1 << 64) - (1 << 33))):
        for b, a in ((2, 2), (3, 7), (40, 900), (M, 1), (0, M)):
            for inv in (False, True):
                check(sc, pat, od, data, b, a, inv, name, base_offset, base_line)
        check(sc, pat, oc, cut, 5, 5, False, name, base_offset, base_line)
        check(sc, pat, oc, cut, 1, 3, True, name, base_offset, base_line)


def test_lines_of_64_mib(api):
    import torch
    sc = api.Scanner(0)
    pat = api.Pattern.load(G.pattern_path("c1"), 0)
    dl = DeviceLines(sc, pat)
    big = b"x" * (64 << 20)
    hit = b"Sherlock Holmes"
    cases = [
        b"a\n" + big + b"\n" + hit + b"\n" + big + b"\nb\n",            # 64 MiB lines before and after the match
        b"a\n" + big + b"\n" + hit + b"\n" + big,                       # ... the last one unterminated
        b"a\nb\n" + big + b" " + hit + b" " + big + b"\nc\nd",          # the selected line itself
        hit + big + b"\nq\n" + big + hit + b"\n",                       # -v: 64 MiB matching lines as context
    ]
    for data in cases:
        dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        for b, a in ((1, 1), (M, M)):
            for inv in (False, True):
                rec, _ = check(sc, pat, dl, dev, b, a, inv, (len(data), b, a))
                if not inv and (b, a) == (1, 1) and data.startswith(b"a\n"):
                    assert len(rec) >= 3 and int(rec["eol"][0]) - int(rec["bol"][0]) in (1, 64 << 20)


def test_config3_never_fires(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c3"), 0)
    op = LO.oracle(cfg("c3"))
    data = corpus.block("c3", 2 << 20)
    for b, a in ((2, 2), (M, M)):
        rec, tot = sc.find_context(pat, data, b, a)
        assert len(rec) == 0 and tot.matches == 0
        rec, tot = check(sc, pat, op, data, b, a, True, "c3")
        assert len(rec) == int((data == 10).sum()) == tot.matches


def test_host_pinned_device_and_misaligned_buffers(api):
    import torch
    sc = api.Scanner(0)
    for name in ("c2", "c4", "w_the"):
        path = cfg(name) if name != "w_the" else G.pattern_path(name)
        pat = api.Pattern.load(path, 0)
        op = LO.oracle(path)
        base = corpus.block("c1" if name == "w_the" else name, 400000)
        dev = torch.from_numpy(base).cuda()
        for lo, hi in ((0, len(base)), (3, 300001), (17, 123457)):
            data = base[lo:hi]
            for inv in (False, True):
                want = CO.find_context(op, data, 2, 3, inv, 1 << 40, 1 << 33)
                for src in (data, dev[lo:hi], torch.from_numpy(data.copy()).pin_memory().numpy()):
                    rec, _ = sc.find_context(pat, src, 2, 3, inv, 1 << 40, 1 << 33)
                    assert rec.tobytes() == want.tobytes(), (name, lo, hi, inv)


def test_overflow_paging_and_argument_checks(api):
    sc = api.Scanner(0)
    L = api.lib()
    pat = api.Pattern.load(cfg("c2"), 0)
    op = LO.oracle(cfg("c2"))
    base = corpus.block("c2", 400000)
    want = CO.find_context(op, base, 2, 2)
    assert len(want) > 10
    out = np.zeros(len(want), dtype=api.LINE_DTYPE)
    cnt = C.c_uint64()
    t = api._Totals()
    args = (sc._h, pat._h, C.c_void_p(base.ctypes.data), len(base), 0, 0)
    rc = L.ugx_find_context(*args, 0, 2, 2, out.ctypes.data, len(want) - 1, C.byref(cnt), C.byref(t))
    assert rc == 5 and cnt.value == len(want)
    paged = np.concatenate([sc.fetch_lines(i, min(7, len(want) - i)) for i in range(0, len(want), 7)])
    assert paged.tobytes() == want.tobytes()
    with pytest.raises(api.UgxError):
        sc.fetch_lines(len(want), 1)
    rc = L.ugx_find_context(*args, 0, 2, 2, out.ctypes.data, len(want), C.byref(cnt), C.byref(t))
    assert rc == 0 and out.tobytes() == want.tobytes()
    assert L.ugx_find_context(*args, 2, 2, 2, out.ctypes.data, len(want), C.byref(cnt), C.byref(t)) == 1
    assert L.ugx_find_context(*args, 0, 2, 2, None, len(want), C.byref(cnt), C.byref(t)) == 1
    dev = C.c_void_p()
    assert L.ugx_find_context_device(*args, 4, 1, 1, C.byref(dev), C.byref(cnt), C.byref(t)) == 1
    assert L.ugx_find_context_device(None, pat._h, C.c_void_p(base.ctypes.data), len(base), 0, 0, 0, 1, 1,
                                     C.byref(dev), C.byref(cnt), C.byref(t)) == 1
    assert L.ugx_find_context_device(*args, 0, 1, 1, C.byref(dev), C.byref(cnt), C.byref(t)) == 0
    assert cnt.value == len(CO.find_context(op, base, 1, 1)) and dev.value


def test_context_records_and_match_records_stay_fetchable_side_by_side(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c5"), 0)
    op = LO.oracle(cfg("c5"))
    a = corpus.block("c5", 1 << 20)
    b = corpus.block("c2", 1 << 20)
    tm = sc.find_all_device(pat, a)
    sc.find_context_device(pat, b, 3, 1, invert=True)
    n = sc.last_lines[1]
    want = CO.find_context(op, b, 3, 1, True)
    assert sc.fetch(0, tm.matches).tobytes() == op.find_all(a).tobytes()
    assert n == len(want) and sc.fetch_lines(0, n).tobytes() == want.tobytes()
    tm = sc.find_all_device(pat, b)
    assert sc.fetch_lines(0, n).tobytes() == want.tobytes()
    assert sc.fetch(0, tm.matches).tobytes() == op.find_all(b).tobytes()


def check_batch(sc, pat, files, b, a, inv, what, op=None, packed=None):
    rec, first, tot = sc.find_context_batch(pat, packed if packed is not None else files, b, a, inv)
    assert len(first) == len(files) + 1 and int(first[0]) == 0 and int(first[-1]) == len(rec), what
    sel = 0
    for i, f in enumerate(files):
        got = rec[int(first[i]):int(first[i + 1])]
        one, t1 = sc.find_context(pat, f, b, a, inv)
        assert got.tobytes() == one.tobytes(), (what, i, b, a, inv, f[:40])
        if op is not None:
            assert got.tobytes() == CO.find_context(op, f, b, a, inv).tobytes(), (what, i)
        sel += t1.matches
    assert tot.matches == sel and tot.newlines == sum(f.count(b"\n") for f in files), (what, tot)
    return rec, first, tot


@pytest.mark.parametrize("name,cname", [("c1", "c1"), ("c2", "c2"), ("c5", "c5"), ("w_the", "c1"), ("empty_line", "c1")])
def test_batch_equals_every_file_alone(api, name, cname):
    sc = api.Scanner(0)
    path = cfg(name) if name in ("c1", "c2", "c5") else G.pattern_path(name)
    pat = api.Pattern.load(path, 0)
    op = LO.oracle(path)
    files = make_files(cname, np.random.default_rng(5), 24) + [b"", b"\n\n", b"x\n"]
    for b, a in ((0, 0), (2, 2), (1, 5), (M, M)):
        for inv in (False, True):
            check_batch(sc, pat, files, b, a, inv, name, op)


def test_batch_context_never_crosses_files(api):
    """files of lines that all match, next to files without a match: no window reaches into a neighbour, also with
    '\\n' as padding between files"""
    import torch
    sc = api.Scanner(0)
    pat = api.Pattern.load(G.pattern_path("c1"), 0)
    hit, miss = b"Sherlock Holmes\n", b"nothing here\n"
    files = [miss * 3, hit, miss * 5 + b"tail", b"", hit + miss, miss, miss + hit * 2, b"\n"]
    for pad in (b"\n", b"X"):
        buf, begins, lens = pack(files, pad)
        for src in (buf, torch.from_numpy(buf).cuda()):
            for b, a in ((2, 2), (M, M)):
                for inv in (False, True):
                    rec, first, _ = check_batch(sc, pat, files, b, a, inv, pad, packed=(src, begins, lens))
                    for i, f in enumerate(files):
                        n = f.count(b"\n") + (1 if f and not f.endswith(b"\n") else 0)
                        assert all(1 <= int(x) <= n for x in rec["line"][int(first[i]):int(first[i + 1])])


def test_batch_of_20000_files(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c2"), 0)
    rng = np.random.default_rng(3)
    base = corpus.block("c2", 8 << 20).tobytes()
    files = []
    for _ in range(20000):
        n = int(rng.integers(0, 4097))
        lo = int(rng.integers(0, len(base) - n))
        files.append(base[lo:lo + n])
    for inv in (False, True):
        rec, first, tot = sc.find_context_batch(pat, files, 2, 2, inv)
        lines, lfirst, ltot = sc.find_lines_batch(pat, files, inv)
        assert tot.matches == ltot.matches and tot.launches <= ltot.launches + 4, (tot, ltot)
        sel = CO.is_selected(rec, inv)
        assert rec[sel].tobytes() == lines.tobytes()
        for i in range(0, 20000, 997):
            one, _ = sc.find_context(pat, files[i], 2, 2, inv)
            assert rec[int(first[i]):int(first[i + 1])].tobytes() == one.tobytes(), i
    rec, first, tot = sc.find_context_batch(pat, [b""] * 100, 2, 2)
    assert len(rec) == 0 and not first.any()
    rec, first, tot = sc.find_context_batch(pat, [], 2, 2)
    assert len(rec) == 0 and list(first) == [0]


def test_batch_overflow_and_argument_checks(api):
    sc = api.Scanner(0)
    L = api.lib()
    pat = api.Pattern.load(cfg("c2"), 0)
    files = make_files("c2", np.random.default_rng(9), 6)
    want, wfirst, _ = sc.find_context_batch(pat, files, 2, 2)
    buf, begins, lens = pack(files)
    first = np.zeros(len(files) + 1, dtype=np.uint64)
    out = np.zeros(len(want), dtype=api.LINE_DTYPE)
    cnt = C.c_uint64()
    t = api._Totals()
    args = (sc._h, pat._h, C.c_void_p(buf.ctypes.data), buf.size, begins.ctypes.data, lens.ctypes.data, len(files))
    rc = L.ugx_find_context_batch(*args, 0, 2, 2, first.ctypes.data, out.ctypes.data, len(want) - 1, C.byref(cnt),
                                  C.byref(t))
    assert rc == 5 and cnt.value == len(want) and np.array_equal(first, wfirst)
    assert sc.fetch_lines(0, len(want)).tobytes() == want.tobytes()
    rc = L.ugx_find_context_batch(*args, 0, 2, 2, first.ctypes.data, out.ctypes.data, len(want), C.byref(cnt),
                                  C.byref(t))
    assert rc == 0 and out.tobytes() == want.tobytes()
    assert L.ugx_find_context_batch(*args, 2, 2, 2, first.ctypes.data, None, 0, C.byref(cnt), C.byref(t)) == 1
    bad = begins.copy()
    bad[1] += 1
    assert L.ugx_find_context_batch(sc._h, pat._h, C.c_void_p(buf.ctypes.data), buf.size, bad.ctypes.data,
                                    lens.ctypes.data, len(files), 0, 2, 2, first.ctypes.data, None, 0, C.byref(cnt),
                                    C.byref(t)) == 1
    assert L.ugx_find_context_batch(*args, 0, 2, 2, None, None, 0, C.byref(cnt), C.byref(t)) == 1
