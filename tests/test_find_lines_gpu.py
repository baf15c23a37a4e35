"""Line records on the GPU (ugx_find_lines*, `ugrep -c` / `ugrep -v` per line): every route against the oracle's
line records (tests/oracle_lines.c) byte for byte, the span route shown to run, BASELINE-sized inputs through size-independent properties,
the edge cases of the carries (lines over thousands of regions, the set-aside last line, hand-over), and the sharded
form against one scan of the whole buffer."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_lib as G
import lines_oracle as LO
import oracle_lib as O
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu
PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")
ROUTES = {"default": {}, "no_span": {"no_span": 1}, "generic": {"force_generic": 1}}
CONFIGS = {"c1": "c1", "c2": "c2", "c3": "c3", "c3b": "c3", "c3c": "c3", "c4": "c4", "c5": "c5"}
EDGE = [b"", b"\n", b"\n\n\n", b"x", b"Sherlock Holmes", b"Sherlock Holmes\n", b"a\r\nSherlock Holmes\r\n\r\nb\r\n",
        b"xSherlock HolmesSherlock Holmes Sherlock Holme\nSherlock Holmes", b"Running\nWalking and Thinking\n\nmorning Singing",
        b"2026-01-02T03:04:05 ERROR svc01 call 555-1234 ext 123-4567 id=1\n" * 3 + b"WARN 111-2222",
        b"a" * 70000 + b" Running ERROR " + b"b" * 70000 + b"\n" + b"Walking WARN"]


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api as A
    return A


def cfg(name):
    return os.path.join(PAT_DIR, name + ".ugxp")


def check(sc, pat, op, data, invert, what, base_offset=0, base_line=0):
    rec, tot = sc.find_lines(pat, data, invert=invert, base_offset=base_offset, base_line=base_line)
    want = op.find_lines(bytes(data) if not isinstance(data, np.ndarray) else data, invert=invert,
                         base_offset=base_offset, base_line=base_line)
    assert len(rec) == len(want) == tot.matches, (what, invert, len(rec), len(want))
    assert rec.tobytes() == want.tobytes(), (what, invert)
    assert tot.flags & 1
    return tot


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
    inputs = [data for _, data in G.cases(name)] + EDGE
    for data in inputs:
        for inv in (False, True):
            tot = check(sc, pat, op, data, inv, (name, route, data[:40]))
            if not inv:
                assert tot.matches == sc.count_lines(pat, data).matches
            assert tot.newlines == data.count(b"\n")
            if route != "default":
                assert tot.kernel == "scan_lines_kernel" or (len(data) == 0 and tot.kernel == "none"), tot


@pytest.mark.parametrize("name", ["c2", "c3b", "c5"])
def test_span_route_runs_where_find_all_takes_the_spans(api, name):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg(name), 0)
    op = LO.oracle(cfg(name))
    data = corpus.block(CONFIGS[name], 4 << 20)
    assert sc.find_all_device(pat, data).kernel == "span_scan_kernel"
    for inv in (False, True):
        tot = check(sc, pat, op, data, inv, name)
        assert tot.kernel == "span_lines_kernel" and not tot.flags & 2, tot


def test_configs_at_baseline_size(api):
    """BASELINE-sized buffers tiled from R copies of one line-aligned block: matching count = count_lines, matching +
    inverted = lines, the block's records repeated with shifted offsets and line numbers (line numbers beyond 2^32
    through base_line; offsets beyond 2^32 in the copies past 4 GiB)"""
    import torch
    sc = api.Scanner(0)
    block_bytes = 32 << 20
    BASE_LINE = (1 << 32) + 3
    for name, gib in (("c1", 4), ("c2", 4), ("c3", 4), ("c3b", 4.75), ("c4", 8), ("c5", 8)):
        pat = api.Pattern.load(cfg(name), 0)
        op = LO.oracle(cfg(name))
        block = corpus.block(CONFIGS[name], block_bytes)
        assert block[-1] == 10
        reps = int(gib * (1 << 30)) // len(block)
        dev = torch.from_numpy(block).cuda().repeat(reps)
        nl = int((block == 10).sum())
        lines_total = reps * nl
        counts = {}
        for inv in (False, True):
            want = op.find_lines(block, invert=inv)
            tot = sc.find_lines_device(pat, dev, invert=inv, base_offset=7, base_line=BASE_LINE)
            assert tot.matches == reps * len(want), (name, inv)
            assert tot.newlines == lines_total
            counts[inv] = tot.matches
            if len(want):
                for r in (0, reps // 2, reps - 1):
                    got = sc.fetch_lines(r * len(want), len(want))
                    for f in ("bol", "eol", "offset"):
                        assert bool(np.all(got[f] == want[f] + r * len(block) + 7)), (name, inv, r, f)
                    assert bool(np.all(got["line"] == want["line"] + r * nl + BASE_LINE)), (name, inv, r)
                    assert bool(np.all(got["len"] == want["len"])) and bool(np.all(got["cap"] == want["cap"]))
                    if r * len(block) > 1 << 32:
                        assert int(got["bol"][0]) > 1 << 32
                assert int(got["line"][-1]) > 1 << 32
        assert counts[False] == sc.count_lines(pat, dev).matches, name
        assert counts[False] + counts[True] == lines_total, name
        del dev
        torch.cuda.empty_cache()


def test_one_line_of_256_mib(api):
    import torch
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c5"), 0)
    op = LO.oracle(cfg("c5"))
    base = corpus.block("c5", 32 << 20).copy()
    base[base == 10] = 32
    big = np.tile(base, 8)
    big[-4:] = np.frombuffer(b" end", dtype=np.uint8)  # unterminated: the line is carried to the buffer end
    dev = torch.from_numpy(big).cuda()
    rec, tot = sc.find_lines(pat, dev)
    assert tot.kernel == "span_lines_kernel" and len(rec) == 1
    assert (int(rec["line"][0]), int(rec["bol"][0]), int(rec["eol"][0])) == (1, 0, len(big))
    first = op.find_all(big[:1 << 20])[0]
    assert (int(rec["offset"][0]), int(rec["len"][0]), int(rec["cap"][0])) == (int(first["offset"]), int(first["len"]), int(first["cap"]))
    rec, _ = sc.find_lines(pat, dev, invert=True)
    assert len(rec) == 0
    # the same line terminated, and a second short line after it
    big2 = np.concatenate([big, np.frombuffer(b"\nno match here\n", dtype=np.uint8)])
    rec, tot = sc.find_lines(pat, torch.from_numpy(big2).cuda(), invert=True)
    assert [(int(r["line"]), int(r["bol"]), int(r["eol"])) for r in rec] == [(2, len(big) + 1, len(big2) - 1)]
    # a 256 MiB line without a match, under -v
    quiet = np.full(256 << 20, ord("x"), dtype=np.uint8)
    quiet[-1] = 10
    rec, tot = sc.find_lines(pat, torch.from_numpy(quiet).cuda(), invert=True)
    assert [(int(r["line"]), int(r["bol"]), int(r["eol"]), int(r["cap"])) for r in rec] == [(1, 0, len(quiet) - 1, 0)]
    assert tot.kernel == "span_lines_kernel"
    rec, _ = sc.find_lines(pat, torch.from_numpy(quiet).cuda())
    assert len(rec) == 0


def test_long_lines_across_regions_against_the_oracle(api):
    """lines straddling many regions, regions without a newline, matches placed at region edges"""
    sc = api.Scanner(0)
    rng = np.random.default_rng(7)
    for name in ("c5", "c2", "c3b"):
        pat = api.Pattern.load(cfg(name), 0)
        op = LO.oracle(cfg(name))
        base = corpus.block(CONFIGS[name], 3 << 20).copy()
        nl = np.flatnonzero(base == 10)
        base[nl[rng.random(len(nl)) < 0.995]] = 32
        for n in (len(base), len(base) - 1, 16384 * 7 + 3, 65536, 65537, 100000):
            for inv in (False, True):
                check(sc, pat, op, base[:n], inv, (name, n))


def test_hand_over_inputs_stay_exact(api):
    sc = api.Scanner(0)
    cases = [
        ("dotstar", b"x" * 20000 + b"a" + b"y" * 40000 + b"b zz a b\n" + b"a b\n" * 10),
        ("pin_pma_lb", b"the s" + b"a" * 1100000 + b"ing sing\nsing song\n"),
        ("dotstar", b"a" + b"q" * 70000 + b"b\n" + b"ab\n" * 5),
        ("c5", b"x" * 100000 + b" ERROR 555-12"),
    ]
    for name, data in cases:
        path = G.pattern_path(name) if name != "c5" else cfg("c5")
        pat = api.Pattern.load(path, 0)
        op = LO.oracle(path)
        for inv in (False, True):
            tot = check(sc, pat, op, data, inv, name)
            assert tot.flags & 2 and tot.kernel == "scan_lines_kernel", (name, tot)


def test_config3_as_named_under_invert_is_every_line(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c3"), 0)
    op = LO.oracle(cfg("c3"))
    data = corpus.block("c3", 2 << 20)
    rec, tot = sc.find_lines(pat, data, invert=True)
    assert len(rec) == int((data == 10).sum()) and tot.kernel == "scan_lines_kernel"
    assert rec.tobytes() == op.find_lines(data, invert=True).tobytes()
    assert len(sc.find_lines(pat, data)[0]) == 0


def test_bases_host_device_misaligned_and_overflow(api):
    import torch
    sc = api.Scanner(0)
    L = api.lib()
    for name in ("c2", "c4", "c5"):
        pat = api.Pattern.load(cfg(name), 0)
        op = LO.oracle(cfg(name))
        base = corpus.block(CONFIGS[name], 400000)
        dev = torch.from_numpy(base).cuda()
        for lo, hi in ((0, len(base)), (3, 300001), (17, 123457)):
            data = base[lo:hi]
            for inv in (False, True):
                want = op.find_lines(data, invert=inv, base_offset=1 << 40, base_line=1 << 33)
                for src in (data, dev[lo:hi], torch.from_numpy(data.copy()).pin_memory().numpy()):
                    rec, _ = sc.find_lines(pat, src, invert=inv, base_offset=1 << 40, base_line=1 << 33)
                    assert rec.tobytes() == want.tobytes(), (name, lo, hi, inv)
        # cap too small: UGX_E_OVERFLOW with the required count; bad flags: UGX_E_INVALID
        want = op.find_lines(base)
        out = np.zeros(len(want), dtype=api.LINE_DTYPE)
        cnt = C.c_uint64()
        t = api._Totals()
        rc = L.ugx_find_lines(sc._h, pat._h, C.c_void_p(base.ctypes.data), len(base), 0, 0, 0, out.ctypes.data,
                              len(want) - 1, C.byref(cnt), C.byref(t))
        assert rc == 5 and cnt.value == len(want)
        rc = L.ugx_find_lines(sc._h, pat._h, C.c_void_p(base.ctypes.data), len(base), 0, 0, 0, out.ctypes.data,
                              len(want), C.byref(cnt), C.byref(t))
        assert rc == 0 and out.tobytes() == want.tobytes()
        rc = L.ugx_find_lines(sc._h, pat._h, C.c_void_p(base.ctypes.data), len(base), 0, 0, 2, out.ctypes.data,
                              len(want), C.byref(cnt), C.byref(t))
        assert rc == 1


def test_line_records_and_match_records_stay_fetchable_side_by_side(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c5"), 0)
    op = LO.oracle(cfg("c5"))
    a = corpus.block("c5", 1 << 20)
    b = corpus.block("c3", 1 << 20)
    tm = sc.find_all_device(pat, a)
    tl = sc.find_lines_device(pat, b, invert=True)
    assert sc.fetch(0, tm.matches).tobytes() == op.find_all(a).tobytes()
    assert sc.fetch_lines(0, tl.matches).tobytes() == op.find_lines(b, invert=True).tobytes()
    tm = sc.find_all_device(pat, b)
    assert sc.fetch_lines(0, tl.matches).tobytes() == op.find_lines(b, invert=True).tobytes()
    assert sc.fetch(0, tm.matches).tobytes() == op.find_all(b).tobytes()
    with pytest.raises(api.UgxError):
        sc.fetch_lines(tl.matches, 1)


@pytest.mark.parametrize("pname,cname", [("c5", "c5"), ("c3b", "c3"), ("c2", "c2"), ("c1", "c1")])
def test_sharded_find_lines_equals_the_single_scan(api, pname, cname):
    import torch
    path = cfg(pname)
    data = corpus.block(cname, 3 << 20)
    sc = api.Scanner(0)
    pat = api.Pattern.load(path, 0)
    lists = [[0], [0, 0], [0, 0, 0]]
    if torch.cuda.device_count() > 1:
        lists.append(list(range(torch.cuda.device_count())))
    for inv in (False, True):
        want, _ = sc.find_lines(pat, data, invert=inv)
        for devs in lists:
            sh = api.Sharded(path, devs)
            rec, tot, info = sh.find_lines(data, invert=inv)
            assert rec.tobytes() == want.tobytes(), (pname, devs, inv)
            assert tot.matches == len(want) and tot.newlines == int((data == 10).sum())
            assert [i["record_base"] for i in info] == list(np.cumsum([0] + [i["matches"] for i in info[:-1]]))
            sh.close()
