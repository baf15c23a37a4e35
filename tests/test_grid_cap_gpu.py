"""Grid-capped parity (scanner option "grid_sms"): every route against the oracle with warps that own many regions.

Nearly every grid-sized launch sizes its grid as min(need, SMs x blocks per SM) and walks the buffer with grid-stride
loops or a region schedule, so on the whole device a warp takes a second 16 KiB region only once the buffer is tens of
MiB.  State carried from one of a warp's regions to the next (span_scan_kernel's probe_tick / via_keep / via_only,
count_lines_stream_kernel's via_tick, RegionSchedule's static rounds, region_begin in the chained launches of the
pipelined host path) is then never checked for exactness at the sizes the CPU oracle can check.  With grid_sms = 1 or 3
the grids are sized as if the device had 1 or 3 SMs, and a buffer of about 10 MiB runs the per-warp schedules a
multi-GiB buffer runs on the full device.  Every capped result must equal the oracle's and the uncapped scan's: records
byte for byte, and matches, newlines, flags and kernel in the totals."""
import os

import numpy as np
import pytest

import bool_oracle as BO
import context_oracle as CO
import golden_lib as G
import lines_oracle as LO
import oracle_lib as O
from test_batch_gpu import make_files
from test_bool_batch import find_lines_bool_batch
from test_gpu_parity import ROUTES as PARITY_ROUTES
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu
PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")

REGION = 16 << 10   # SC_REGION: the unit of RegionSchedule and of the span kernels' grid-stride loop over regions
SPAN = 512          # a span kernel's span, and the window a region takes its chain state from
# Size rule.  An SM holds at most 64 resident warps (2048 threads), so at grid_sms = 1 no launch has more than 64 warps.
# A buffer of 64 x 9 regions then gives every warp of every region-based kernel at least 9 regions: one full probe_tick
# cycle of span_scan_kernel (a probe every 8th region) plus one region, at least 9 x 32 = 288 spans for
# count_lines_stream_kernel's probe every 64th span, and static rounds in RegionSchedule ((576 - 72) / 64 = 7 rounds).
MAX_WARPS_PER_SM = 64
MIN_REGIONS_PER_WARP = 9
MIN_BYTES = MAX_WARPS_PER_SM * MIN_REGIONS_PER_WARP * REGION  # 9 MiB
# three CTAs keep the round-robin from lining up with power-of-two region counts; 0 is the device's own grid (control)
CAPS = (1, 3)
ROUTES = dict(PARITY_ROUTES, no_search={"no_search": 1})
# the calls each route changes: "lines" count_lines, "matches" count_matches, "list" find_all, "hit" / "miss" find_lines
ROUTE_CALLS = {"default": ("lines", "matches", "list", "hit", "miss"), "generic": ("lines", "matches", "list", "hit", "miss"),
               "no_span": ("lines", "matches", "list", "hit", "miss"), "legacy_any": ("lines",), "stream": ("lines",),
               "stream_nl": ("lines",), "two_pass": ("list",), "match_lines": ("lines", "matches"), "no_search": ("lines",)}
ALL_CALLS = ("lines", "matches", "list", "hit", "miss")
TOT_NEWLINES, TOT_SPAN_HANDOVER = 1, 2


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api as A
    return A


def cfg(name):
    return os.path.join(PAT_DIR, name + ".ugxp")


def totals_key(t):
    return (t.matches, t.newlines, t.flags, t.kernel)


def check_records(got, want, what):
    """byte-for-byte equality, reporting the first differing record and the region it lies in"""
    if len(got) == len(want) and got.tobytes() == want.tobytes():
        return
    n = min(len(got), len(want))
    diff = np.flatnonzero(got[:n] != want[:n])
    i = int(diff[0]) if len(diff) else n
    at = got[i] if i < len(got) else want[i]
    raise AssertionError("%r: %d records, want %d; first difference at record %d (offset %d, region %d): %r vs %r" % (
        what, len(got), len(want), i, int(at["offset"]), int(at["offset"]) // REGION,
        got[i] if i < len(got) else None, want[i] if i < len(want) else None))


def call(sc, pat, data, kind):
    """-> (records or None, totals)"""
    if kind == "lines":
        return None, sc.count_lines(pat, data)
    if kind == "matches":
        return None, sc.count_matches(pat, data)
    if kind == "list":
        return sc.find_all(pat, data)
    return sc.find_lines(pat, data, invert=kind == "miss")


def at_caps(sc, run, want, what, nl=None, count=None):
    """run() at the device's own grid and at every cap: each result equals `want` (a count, or records whose count is
    len(want) unless given) and the uncapped one (records, and matches / newlines / flags / kernel of the totals)"""
    out = {}
    try:
        for k in (0,) + CAPS:
            sc.set_option("grid_sms", k)
            out[k] = run()
    finally:
        sc.set_option("grid_sms", 0)
    for k, (rec, tot) in out.items():
        w = (what, "grid_sms=%d" % k)
        if rec is None:
            assert tot.matches == want, (w, tot, want)
        else:
            check_records(rec, want, w)
            assert tot.matches == (len(want) if count is None else count), (w, tot)
        if nl is not None and tot.flags & TOT_NEWLINES:
            assert tot.newlines == nl, (w, tot, nl)
        if k:
            assert totals_key(tot) == totals_key(out[0][1]), (w, tot, out[0][1])
    return out


class Oracle:
    """the oracle's answers for one buffer, each computed once"""

    def __init__(self, path, data):
        self.op, self.data, self.memo = LO.oracle(path), data, {}

    def want(self, kind):
        if kind not in self.memo:
            op, d = self.op, self.data
            self.memo[kind] = (op.count_lines(d) if kind == "lines" else op.count_matches(d) if kind == "matches"
                               else op.find_all(d) if kind == "list" else op.find_lines(d, kind == "miss"))
        return self.memo[kind]

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        assert data is self.data and base_offset == 0 and base_line == 0
        return self.want("miss" if invert else "hit")


# ---- 1. every golden pattern through every route ----

def splice_sites(texts, nregions, rng):
    """(position, text, framed) of every case text at region-relative offsets 0, 1, 15, 16, 511, 512, 513, REGION - len,
    REGION - 1 (across the next region start), across the region start from inside the window before it, and inside that
    window; each site in a region of its own past the first 200, so in a later region of its warp at every cap"""
    regions = rng.permutation(np.arange(200, nregions - 2))
    sites, j = [], 0
    for t in texts:
        L = len(t)
        for rel in (0, 1, 15, 16, 511, 512, 513, REGION - L, REGION - 1, -(L // 2) - 1, -SPAN + 3):
            sites.append((int(regions[j % len(regions)]) * REGION + rel, t, j % 2 == 0))
            j += 1
    return sites


_golden_input = None


def golden_input():
    """about 10 MiB of corpus text (2 MiB blocks of c1..c5), three lines of 20 KiB across two region starts each (in
    later regions of their warps), and every golden edge case text spliced in at the sites above, every other one on
    lines of its own.  The long lines are no longer: the line-at-a-time kernels attempt a pattern like `a.*b` at every
    candidate of a line up to its end, so their cost grows with the square of the line length."""
    global _golden_input
    if _golden_input is None:
        base = np.concatenate([corpus.block(c, 2 << 20) for c in ("c1", "c2", "c3", "c4", "c5")])
        nregions = len(base) // REGION
        for q in (260, 400, 610):
            lo, hi = q * REGION - 3000, q * REGION - 3000 + (20 << 10)
            seg = base[lo:hi]
            seg[seg == 10] = ord(" ")
        texts = sorted({bytes(d) for c, d in (x for n in G.pattern_names() for x in G.cases(n))
                        if c["input"][0] == "edge" and 0 < len(d) <= 4096})
        for at, t, framed in splice_sites(texts, nregions, np.random.default_rng(17)):
            base[at:at + len(t)] = np.frombuffer(t, dtype=np.uint8)
            if framed:
                base[at - 1] = base[at + len(t)] = 10
        _golden_input = base
    return _golden_input


def load_or_skip(api, path):
    try:
        return api.Pattern.load(path, 0)
    except api.UgxError as ex:
        assert ex.code == 2, ex  # UGX_E_UNSUPPORTED: outside the path's scope, rejected loudly
        pytest.skip("out of scope: %s" % ex)


@pytest.mark.parametrize("name", G.pattern_names())
def test_golden_pattern_every_route(api, name):
    import torch
    pat = load_or_skip(api, G.pattern_path(name))
    data = golden_input()
    assert len(data) >= MIN_BYTES
    dev = torch.from_numpy(data).cuda()
    ora = Oracle(G.pattern_path(name), data)
    nl = int((data == 10).sum())
    for route, opts in ROUTES.items():
        sc = api.Scanner(0)
        for k, v in opts.items():
            sc.set_option(k, v)
        for kind in ROUTE_CALLS[route]:
            at_caps(sc, lambda: call(sc, pat, dev, kind), ora.want(kind), (name, route, kind), nl)


# ---- 2. config patterns and library-compiled patterns, with the candidate predicate always evaluated and without the
# search automaton ----

def w3000_path(api, tmp_path, icase=False, count=3000):
    words = corpus.words_list(11, count)
    opc, pf = api.compile_words(words, icase)
    path = str(tmp_path / ("w%d%s.ugxp" % (count, "i" if icase else "")))
    api.write_ugxp(path, opc, pf)
    return words, path


def config_pattern(api, tmp_path, name):
    """(device pattern, oracle pattern file, corpus)"""
    if name in ("c1", "c2", "c3", "c4", "c5"):
        return api.Pattern.load(cfg(name), 0), cfg(name), name
    if name == "c2s":
        return api.Pattern.load(cfg("c2"), 0), cfg("c2"), "c2s"
    if name == "c3c":
        return api.Pattern.load(cfg("c3c"), 0), cfg("c3c"), "c3"
    if name == "literal":
        return api.Pattern.literal(b"Sherlock Holmes", 0), cfg("c1"), "c1"
    if name == "words":
        return api.Pattern.words(corpus.words_list(), 0), cfg("c2"), "c2"
    if name == "words_i":
        words, path = w3000_path(api, tmp_path, icase=True, count=1000)
        return api.Pattern.words(words, 0, icase=True), path, "c2"
    words, path = w3000_path(api, tmp_path)
    pat = api.Pattern.words(words, 0)
    assert pat.info["table_in_smem"] == 0  # the table stays in global memory: the span kernel runs at 256 threads
    return pat, path, "c2"


CONFIGS = ["c1", "c2", "c2s", "c3", "c3c", "c4", "c5", "literal", "words", "words_i", "w3000"]


@pytest.mark.parametrize("name", CONFIGS)
def test_config_every_mode(api, tmp_path, name):
    """12 MiB blocks, every call, on the default route, with no_cover (the lazy, mask and via_only forms of the span
    kernel and the stream kernel's probe evaluate the predicate) and with no_search (count_lines_stream_kernel)"""
    import torch
    pat, path, cname = config_pattern(api, tmp_path, name)
    data = corpus.block(cname, 12 << 20)
    dev = torch.from_numpy(data).cuda()
    ora = Oracle(path, data)
    nl = int((data == 10).sum())
    for opts in ({}, {"no_cover": 1}, {"no_search": 1}):
        sc = api.Scanner(0)
        for k, v in opts.items():
            sc.set_option(k, v)
        for kind in ALL_CALLS:
            at_caps(sc, lambda: call(sc, pat, dev, kind), ora.want(kind), (name, opts, kind), nl)


# ---- 3. line stages ----

def long_lines(data, rng, count=6, length=40 << 10):
    out = data.copy()
    for lo in rng.integers(64 * REGION, len(data) - length, size=count):
        seg = out[lo:lo + length]
        seg[seg == 10] = ord(" ")
    return out


@pytest.mark.parametrize("name", ["c2", "c5"])
def test_context_lines(api, name):
    data = long_lines(corpus.block(name, 10 << 20), np.random.default_rng(3))
    pat = api.Pattern.load(cfg(name), 0)
    ora = Oracle(cfg(name), data)
    sc = api.Scanner(0)
    for before, after in ((0, 2), (3, 0), (2, 2)):
        for inv in (False, True):
            want = CO.find_context(ora, data, before, after, inv)
            at_caps(sc, lambda: sc.find_context(pat, data, before, after, invert=inv), want, (name, before, after, inv),
                    count=int(CO.is_selected(want, inv).sum()))


def literal_term(api, tmp_path, text):
    opc, pf = api.compile_literal(text)
    path = str(tmp_path / ("lit_%s.ugxp" % text.hex()))
    api.write_ugxp(path, opc, pf)
    return api.Pattern.literal(text, 0), path


def test_bool_lines(api, tmp_path):
    """--and, --andnot and a three-term CNF, both polarities, find and count"""
    data = long_lines(corpus.block("c5", 10 << 20), np.random.default_rng(4))
    pats, oras = [api.Pattern.load(cfg("c5"), 0)], [Oracle(cfg("c5"), data)]
    for text in (b"ERROR", b"555"):
        p, path = literal_term(api, tmp_path, text)
        pats.append(p)
        oras.append(Oracle(path, data))
    sc = api.Scanner(0)
    for cnf in ([[0], [1]], [[0], [~1]], [[1, 2], [~0]], [[0, 1, 2], [~2]]):
        for inv in (False, True):
            want = BO.find_lines_bool(oras, cnf, data, inv)
            out = at_caps(sc, lambda: sc.find_lines_bool(pats, cnf, data, inv), want, ("bool", cnf, inv))
            assert all(t.kernel == "bool_count_kernel" for _, t in out.values())
            at_caps(sc, lambda: (None, sc.count_lines_bool(pats, cnf, data, inv)), len(want), ("bool -c", cnf, inv))


def test_check_text_and_count_newlines(api):
    base = corpus.block("c4", 11 << 20)
    bad = base.copy()
    bad[600 * REGION + 77] = 0xff                  # not UTF-8, in a later region of its warp
    nul = base.copy()
    nul[640 * REGION - 1] = 0
    sc = api.Scanner(0)
    for src in (base, bad, nul):
        for n in [k * REGION + d for k in (576, 577, 640, 673) for d in (-17, -1, 0, 1, 15)] + [len(src)]:
            data = src[:n]
            want = (O.isutf8(data), O.has_nul(data))
            nl = int((data == 10).sum())
            for k in (0,) + CAPS:
                sc.set_option("grid_sms", k)
                t = sc.check_text(data)
                assert (t["is_utf8"], t["has_nul"]) == want, (n, k)
                assert sc.count_newlines(data).newlines == nl, (n, k)
            sc.set_option("grid_sms", 0)


# ---- 4. the batch forms ----

class Memo:
    """an oracle's answers per file, computed once"""

    def __init__(self, path):
        self.op, self.memo = LO.oracle(path), {}

    def get(self, kind, f):
        key = (kind, bytes(f))
        if key not in self.memo:
            op = self.op
            self.memo[key] = (op.count_lines(f) if kind == "lines" else op.count_matches(f) if kind == "matches"
                              else op.find_all(f) if kind == "list" else op.find_lines(f, kind == "miss"))
        return self.memo[key]

    def find_lines(self, data, invert=False, base_offset=0, base_line=0):
        assert base_offset == 0 and base_line == 0
        return self.get("miss" if invert else "hit", data)


def per_file(files, fn):
    """records of every file alone, concatenated in file order, and first[]"""
    per = [fn(f) for f in files]
    first = np.zeros(len(files) + 1, dtype=np.uint64)
    first[1:] = np.cumsum([len(r) for r in per], dtype=np.uint64)
    return np.concatenate(per), first


def check_batch(rec, first, want, wfirst, files, what):
    assert np.array_equal(first, wfirst), what
    if rec.tobytes() != want.tobytes():
        for i in range(len(files)):
            check_records(rec[int(first[i]):int(first[i + 1])], want[int(wfirst[i]):int(wfirst[i + 1])], (what, "file", i))
        raise AssertionError(what)


BATCH_CNFS = ([[0], [~1]], [[1, 2], [0]])


def test_batch_forms(api, tmp_path):
    """about 3 000 files of the make_files kind (empty, 1 byte, 16383 / 16384 / 16385 bytes, up to 70 000 bytes, cut
    anywhere): every file's slice against the oracle's scan of that file alone"""
    files = make_files("c5", np.random.default_rng(23), 3000)
    assert sum(map(len, files)) >= MIN_BYTES
    pat = api.Pattern.load(cfg("c5"), 0)
    memo = Memo(cfg("c5"))
    pats, memos = [pat], [memo]
    for text in (b"WARN", b"555"):
        p, path = literal_term(api, tmp_path, text)
        pats.append(p)
        memos.append(Memo(path))
    nl = sum(f.count(b"\n") for f in files)
    counts = {mode: [memo.get(mode, f) for f in files] for mode in ("lines", "matches")}
    records = {"list": per_file(files, lambda f: memo.get("list", f))}
    for inv in (False, True):
        records["lines", inv] = per_file(files, lambda f: memo.get("miss" if inv else "hit", f))
        records["context", inv] = per_file(files, lambda f: CO.find_context(memo, f, 2, 1, inv))
        for cnf in BATCH_CNFS:
            records["bool", str(cnf), inv] = find_lines_bool_batch(memos, cnf, files, inv)
    sc = api.Scanner(0)
    try:
        for k in (0,) + CAPS:
            sc.set_option("grid_sms", k)
            for mode in ("lines", "matches"):
                got, tot = sc.count_batch(pat, files, mode)
                assert list(map(int, got)) == counts[mode], (k, mode)
            rec, first, tot = sc.find_all_batch(pat, files)
            check_batch(rec, first, *records["list"], files, (k, "find_all_batch"))
            for inv in (False, True):
                rec, first, tot = sc.find_lines_batch(pat, files, inv)
                check_batch(rec, first, *records["lines", inv], files, (k, "find_lines_batch", inv))
                rec, first, tot = sc.find_context_batch(pat, files, 2, 1, inv)
                check_batch(rec, first, *records["context", inv], files, (k, "find_context_batch", inv))
                for cnf in BATCH_CNFS:
                    want, wfirst, wcounts = records["bool", str(cnf), inv]
                    rec, first, tot = sc.find_lines_bool_batch(pats, cnf, files, inv)
                    check_batch(rec, first, want, wfirst, files, (k, "find_lines_bool_batch", cnf, inv))
                    assert tot.newlines == nl, (k, tot)
                    got, ct = sc.count_lines_bool_batch(pats, cnf, files, inv)
                    assert np.array_equal(got, wcounts) and ct.matches == len(want), (k, cnf, inv)
    finally:
        sc.set_option("grid_sms", 0)


# ---- 5. chained launches of the pipelined host path ----

# (pattern, corpus, options, a match to put across each chunk edge, whether the pinned buffer takes chained launches: c4's
# longest match is unbounded, so it is copied whole and scanned in one launch)
CHAINED = [("c1", "c1", {}, b"Sherlock Holmes", True), ("c2", "c2", {}, None, True),
           ("c2", "c2", {"no_search": 1}, None, True), ("c4", "c4", {}, "naïve".encode(), False)]


@pytest.mark.parametrize("pname,cname,opts,needle,chained", CHAINED, ids=["c1", "c2", "c2_no_search", "c4"])
def test_chained_launches(api, pname, cname, opts, needle, chained):
    """75 MiB of page-locked host memory at grid_sms = 1: each 32 MiB chunk's launch has static rounds and
    region_begin != 0, and a match lies across each chunk edge.  The count equals the uncapped device-resident scan and
    the oracle's count of the whole buffer; the pageable (feeder) path once as well."""
    import torch
    pat = api.Pattern.load(cfg(pname), 0)
    op = O.OraclePattern(cfg(pname))
    host = np.tile(corpus.block(cname, 5 << 20), 15)
    if needle is None:
        needle = corpus.words_list()[0]
    for edge in (32 << 20, 64 << 20):
        at = edge - len(needle) // 2
        host[at - 1] = host[at + len(needle)] = 10
        host[at:at + len(needle)] = np.frombuffer(needle, dtype=np.uint8)
    want = op.count_lines(host)
    sc = api.Scanner(0)
    for k, v in opts.items():
        sc.set_option(k, v)
    ctrl = sc.count_lines(pat, torch.from_numpy(host).cuda())
    assert ctrl.matches == want, (pname, opts, ctrl, want)
    pinned = torch.from_numpy(host).pin_memory()
    sc.set_option("grid_sms", 1)
    got = sc.count_lines(pat, pinned.numpy())
    assert got.launches >= 3 if chained else got.launches == 1, got
    assert totals_key(got) == totals_key(ctrl), (pname, opts, got, ctrl)
    got = sc.count_lines(pat, host)
    assert got.launches == 1 and totals_key(got) == totals_key(ctrl), (pname, opts, "pageable", got, ctrl)


# ---- 6. hand-over under the cap ----

def test_hand_over_under_the_cap(api):
    """the inputs of test_gpu_parity's hand-over test, and a long line in which a match longer than a window straddles
    the start of region 100 (a later region of its warp at every cap): UGX_TOT_SPAN_HANDOVER, and exact results"""
    prefix = corpus.block("c1", 100 * REGION - 25000)
    prefix = prefix[:np.flatnonzero(prefix == 10)[-1] + 1].tobytes()
    pad = 100 * REGION - 25000 - len(prefix)
    straddle = prefix + b"x" * (20000 + pad) + b"a" + b"y" * 40000 + b"b zz a b\n" + corpus.block("c1", 1 << 20).tobytes()
    assert straddle.index(b"a" + b"y" * 10) < 100 * REGION < straddle.index(b"yb zz")
    cases = [
        ("dotstar", b"x" * 20000 + b"a" + b"y" * 40000 + b"b zz a b\n" + b"a b\n" * 10),
        ("pin_pma_lb", b"the s" + b"a" * 1100000 + b"ing sing\nsing song\n"),
        ("dotstar", b"a" + b"q" * 70000 + b"b\n" + b"ab\n" * 5),
        ("c5", b"x" * 100000 + b" ERROR 555-12"),
        ("dotstar", straddle),
    ]
    sc = api.Scanner(0)
    for name, data in cases:
        path = G.pattern_path(name) if name != "c5" else cfg("c5")
        pat = api.Pattern.load(path, 0)
        op = O.OraclePattern(path)
        out = at_caps(sc, lambda: sc.find_all(pat, data), op.find_all(data), (name, len(data)))
        for rec, tot in out.values():
            assert tot.flags & TOT_SPAN_HANDOVER and tot.kernel != "span_scan_kernel", (name, tot)
        out = at_caps(sc, lambda: (None, sc.count_matches(pat, data)), op.count_matches(data), (name, len(data)),
                      data.count(b"\n"))
        for _, tot in out.values():
            assert tot.flags & TOT_NEWLINES, (name, tot)


# ---- 7. the option itself ----

def test_the_option(api):
    import torch
    pat = api.Pattern.load(cfg("c5"), 0)
    data = corpus.block("c5", 10 << 20)
    dev = torch.from_numpy(data).cuda()
    want = O.OraclePattern(cfg("c5")).find_all(data)
    sc = api.Scanner(0)
    with pytest.raises(api.UgxError) as ex:
        sc.set_option("grid_sms", -1)
    assert ex.value.code == 1
    with pytest.raises(api.UgxError) as ex:
        sc.set_option("grid_smz", 1)
    assert ex.value.code == 1
    for k in (0, 1, 100000, 0, 3, 0):
        sc.set_option("grid_sms", k)
        rec, tot = sc.find_all(pat, dev)
        check_records(rec, want, ("grid_sms", k))
        assert tot.kernel == "span_scan_kernel" and not tot.flags & TOT_SPAN_HANDOVER, (k, tot)
    sh = api.Sharded(cfg("c5"), [0, 0])
    with pytest.raises(api.UgxError):
        sh.set_option("grid_sms", -1)
    sh.set_option("grid_sms", 1)
    tot, rec, info = sh.scan(data, "records", cap=len(want) + 10)
    check_records(rec, want, "sharded [0, 0] at grid_sms=1")
    assert tot.matches == len(want) and tot.newlines == int((data == 10).sum())
    sh.close()
