"""Match and line records of many files in one launch sequence (ugx_find_all_batch, ugx_find_lines_batch): file i's
slice rec[first[i]:first[i + 1]] must be byte for byte what the oracle returns for file i scanned ALONE (offsets from
the file's start, line numbers from 1), in both polarities of the line records; plus the per-file counts against
ugx_count_batch, the padding between files, a long line inside a batch, config 3, a source tree's worth of files,
host / pinned / device buffers, the two record arenas side by side, and the argument checks."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_lib as G
import lines_oracle as LO
import oracle_lib as O
from test_batch_gpu import make_files
from test_find_lines_gpu import EDGE
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu
PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")
CONFIGS = {"c1": "c1", "c2": "c2", "c3": "c3", "c3b": "c3", "c4": "c4", "c5": "c5"}


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api as A
    return A


def cfg(name):
    return os.path.join(PAT_DIR, name + ".ugxp")


def pack(files, pad=b"X"):
    """the files on 16-byte boundaries, the gaps (and 16 bytes after the last file) filled by repeating `pad`"""
    begins, at = [], 0
    for f in files:
        begins.append(at)
        at = (at + len(f) + 15) & ~15
    total = at + 16
    buf = np.frombuffer((pad * (total // len(pad) + 1))[:total], dtype=np.uint8).copy()
    for b, f in zip(begins, files):
        buf[b:b + len(f)] = np.frombuffer(bytes(f), dtype=np.uint8)
    return buf, np.array(begins, dtype=np.uint64), np.array([len(f) for f in files], dtype=np.uint64)


def raw(api, sc, pat, buf, begins, lens, lines, flags=0, cap=0, out=None, first=True, nfiles=None):
    """one ugx_find_{all,lines}_batch call through the C ABI: (rc, n_out, first, totals, out)"""
    L = api.lib()
    nfiles = len(lens) if nfiles is None else nfiles
    fst = np.full(nfiles + 1, 77, dtype=np.uint64)
    cnt = C.c_uint64(99)
    t = api._Totals()
    ptr = buf.data_ptr() if hasattr(buf, "data_ptr") else buf.ctypes.data
    nbytes = buf.numel() if hasattr(buf, "numel") else buf.size
    args = [sc._h, pat._h, C.c_void_p(ptr), nbytes, begins.ctypes.data, lens.ctypes.data, nfiles]
    if lines:
        args.append(flags)
    args += [fst.ctypes.data if first else None, out.ctypes.data if out is not None else None, cap, C.byref(cnt),
             C.byref(t)]
    rc = (L.ugx_find_lines_batch if lines else L.ugx_find_all_batch)(*args)
    return rc, cnt.value, fst, t, out


def line_count(f):
    return f.count(b"\n") + (1 if len(f) and not f.endswith(b"\n") else 0)


def check_against_oracle(sc, pat, op, files, what):
    """all three record forms of the batch against the oracle on every file alone"""
    rec, first, tot = sc.find_all_batch(pat, files)
    assert len(first) == len(files) + 1 and int(first[0]) == 0 and int(first[-1]) == len(rec) == tot.matches, what
    for i, f in enumerate(files):
        assert rec[int(first[i]):int(first[i + 1])].tobytes() == op.find_all(f).tobytes(), (what, "matches", i, f[:40])
    assert tot.newlines == sum(f.count(b"\n") for f in files) and tot.flags & 1, what
    if any(len(f) for f in files):
        assert tot.kernel == "scan_batch_kernel" and 2 <= tot.launches <= 3, (what, tot)
    for inv in (False, True):
        rec, first, tot = sc.find_lines_batch(pat, files, invert=inv)
        assert int(first[-1]) == len(rec) == tot.matches, (what, inv)
        for i, f in enumerate(files):
            want = op.find_lines(f, invert=inv)
            assert rec[int(first[i]):int(first[i + 1])].tobytes() == want.tobytes(), (what, inv, i, f[:40])
        assert tot.newlines == sum(f.count(b"\n") for f in files) and tot.flags & 1, what


@pytest.mark.parametrize("name", G.pattern_names())
def test_golden_patterns_file_by_file(api, name):
    sc = api.Scanner(0)
    try:
        pat = api.Pattern.load(G.pattern_path(name), 0)
    except api.UgxError as ex:
        assert ex.code == 2, ex
        pytest.skip("out of scope: %s" % ex)
    op = LO.oracle(G.pattern_path(name))
    inputs = [bytes(data) for _, data in G.cases(name)]
    files = inputs + list(EDGE) + [b"", b"\n"]
    for data in inputs:
        files += [data[:1], data[:15], data[:16], data[:17]]
    check_against_oracle(sc, pat, op, files, name)


@pytest.mark.parametrize("name", ["c1", "c2", "c3b", "c4", "c5"])
def test_config_patterns_on_random_cuts(api, name):
    """cuts of 16383 / 16384 / 16385 / 40000 / 70000 bytes: lines cross tile edges inside one file"""
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg(name), 0)
    op = LO.oracle(cfg(name))
    files = make_files(CONFIGS[name], np.random.default_rng(11), 60)
    check_against_oracle(sc, pat, op, files, name)
    per_lines, _ = sc.count_batch(pat, files, "lines")
    per_matches, _ = sc.count_batch(pat, files, "matches")
    _, fm, _ = sc.find_all_batch(pat, files)
    _, fl, tl = sc.find_lines_batch(pat, files)
    _, fv, tv = sc.find_lines_batch(pat, files, invert=True)
    assert list(np.diff(fm)) == list(per_matches), name
    assert list(np.diff(fl)) == list(per_lines), name
    assert list(np.diff(fl) + np.diff(fv)) == [line_count(f) for f in files], name
    assert tl.newlines == tv.newlines == sum(f.count(b"\n") for f in files)


@pytest.mark.parametrize("pad", [b"\n", b"ERROR\n", b"Sherlock Holmes\n"])
def test_padding_between_files_is_never_text(api, pad):
    sc = api.Scanner(0)
    for name in ("c5", "c1", "bol"):
        path = cfg(name) if os.path.exists(cfg(name)) else G.pattern_path(name)
        pat = api.Pattern.load(path, 0)
        files = make_files("c5" if name != "c1" else "c1", np.random.default_rng(5), 30)
        files += [b"ERROR", b"ERR", b"Sherlock", b"x\n", b"\nERROR 1"]
        neutral, begins, lens = pack(files)
        padded, begins2, lens2 = pack(files, pad)
        assert (begins == begins2).all() and (lens == lens2).all()
        for lines, flags in ((False, 0), (True, 0), (True, 1)):
            want = raw(api, sc, pat, neutral, begins, lens, lines, flags, cap=1 << 18,
                       out=np.zeros(1 << 18, dtype=api.LINE_DTYPE if lines else api.MATCH_DTYPE))
            got = raw(api, sc, pat, padded, begins, lens, lines, flags, cap=1 << 18,
                      out=np.zeros(1 << 18, dtype=api.LINE_DTYPE if lines else api.MATCH_DTYPE))
            assert want[0] == got[0] == 0
            assert want[1] == got[1] and (want[2] == got[2]).all(), (name, pad, lines, flags)
            assert want[4][:want[1]].tobytes() == got[4][:got[1]].tobytes(), (name, pad, lines, flags)
            assert want[3].newlines == got[3].newlines == sum(f.count(b"\n") for f in files)


def test_a_long_line_in_the_middle_of_small_files(api):
    """a 1 MiB file with one 300 KB line (matches at both ends) among small files"""
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c5"), 0)
    op = LO.oracle(cfg("c5"))
    big = corpus.block("c5", 1 << 20).copy()
    lo = 400000
    seg = big[lo:lo + 300000]
    seg[seg == 10] = 32
    big[lo - 1] = 10
    big[lo + 300000] = 10
    big[lo:lo + 6] = np.frombuffer(b"ERROR ", dtype=np.uint8)
    big[lo + 300000 - 6:lo + 300000] = np.frombuffer(b" ERROR", dtype=np.uint8)
    base = corpus.block("c5", 200000).tobytes()
    files = [base[i * 997:i * 997 + 300 + i] for i in range(40)]
    files = files[:20] + [big.tobytes()] + files[20:]
    check_against_oracle(sc, pat, op, files, "long line")
    rec, first, _ = sc.find_lines_batch(pat, files)
    mine = rec[int(first[20]):int(first[21])]
    row = mine[np.flatnonzero(mine["bol"] == lo)]
    assert len(row) == 1 and int(row["eol"][0]) == lo + 300000 and int(row["offset"][0]) == lo


def test_config3_never_matches_and_inverts_to_every_line(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c3"), 0)
    op = LO.oracle(cfg("c3"))
    files = make_files("c3", np.random.default_rng(4), 40)
    rec, first, tot = sc.find_all_batch(pat, files)
    assert len(rec) == 0 and int(first[-1]) == 0 and tot.newlines == sum(f.count(b"\n") for f in files)
    rec, first, _ = sc.find_lines_batch(pat, files)
    assert len(rec) == 0
    rec, first, tot = sc.find_lines_batch(pat, files, invert=True)
    assert len(rec) == sum(line_count(f) for f in files) == tot.matches
    for i, f in enumerate(files):
        assert rec[int(first[i]):int(first[i + 1])].tobytes() == op.find_lines(f, invert=True).tobytes(), i


def test_a_source_tree_worth_of_files(api):
    """20 000 files of up to 4 KiB: at most three launches, per-file ranges against count_batch and the oracle"""
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c5"), 0)
    op = LO.oracle(cfg("c5"))
    base = corpus.block("c5", 2 << 20).tobytes()
    rng = np.random.default_rng(8)
    files = []
    for _ in range(20000):
        lo = int(rng.integers(0, len(base) - 4096))
        files.append(base[lo:lo + int(rng.integers(0, 4096))])
    idx = rng.integers(0, len(files), size=300)
    counts, _ = sc.count_batch(pat, files, "matches")
    rec, first, tot = sc.find_all_batch(pat, files)
    assert tot.launches <= 3 and int(first[-1]) == tot.matches == int(counts.sum())
    for i in idx:
        assert rec[int(first[i]):int(first[i + 1])].tobytes() == op.find_all(files[i]).tobytes(), i
    counts, _ = sc.count_batch(pat, files, "lines")
    for inv in (False, True):
        rec, first, tot = sc.find_lines_batch(pat, files, invert=inv)
        assert tot.launches <= 3
        if not inv:
            assert int(first[-1]) == tot.matches == int(counts.sum())
        for i in idx:
            assert rec[int(first[i]):int(first[i + 1])].tobytes() == op.find_lines(files[i], invert=inv).tobytes(), i


def test_host_pinned_and_device_buffers_agree(api):
    import torch
    sc = api.Scanner(0)
    for name in ("c2", "c5"):
        pat = api.Pattern.load(cfg(name), 0)
        files = make_files(CONFIGS[name], np.random.default_rng(9), 40)
        buf, begins, lens = pack(files)
        sources = [buf, torch.from_numpy(buf.copy()).pin_memory().numpy(), torch.from_numpy(buf).cuda()]
        for lines, flags in ((False, 0), (True, 0), (True, 1)):
            dt = api.LINE_DTYPE if lines else api.MATCH_DTYPE
            res = [raw(api, sc, pat, src, begins, lens, lines, flags, cap=1 << 18, out=np.zeros(1 << 18, dtype=dt))
                   for src in sources]
            for rc, n, fst, t, out in res:
                assert rc == 0 and n == res[0][1] and (fst == res[0][2]).all(), (name, lines, flags)
                assert out[:n].tobytes() == res[0][4][:n].tobytes(), (name, lines, flags)
            rec, first, _ = (sc.find_lines_batch(pat, files, invert=bool(flags)) if lines else sc.find_all_batch(pat, files))
            assert rec.tobytes() == res[0][4][:res[0][1]].tobytes() and (first == res[0][2]).all()


def test_match_and_line_arenas_stay_valid_side_by_side(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c5"), 0)
    op = LO.oracle(cfg("c5"))
    a = corpus.block("c5", 1 << 20)
    files = make_files("c5", np.random.default_rng(12), 30)
    buf, begins, lens = pack(files)
    tm = sc.find_all_device(pat, a)
    rc, n, first, _, _ = raw(api, sc, pat, buf, begins, lens, True)  # device only
    assert rc == 0 and n == int(first[-1])
    assert sc.fetch(0, tm.matches).tobytes() == op.find_all(a).tobytes()
    for i, f in enumerate(files):
        got = sc.fetch_lines(int(first[i]), int(first[i + 1] - first[i]))
        assert got.tobytes() == op.find_lines(f).tobytes(), i
    tl = sc.find_lines_device(pat, a, invert=True)
    rc, n, first, _, _ = raw(api, sc, pat, buf, begins, lens, False)
    assert rc == 0 and n == int(first[-1])
    assert sc.fetch_lines(0, tl.matches).tobytes() == op.find_lines(a, invert=True).tobytes()
    for i, f in enumerate(files):
        assert sc.fetch(int(first[i]), int(first[i + 1] - first[i])).tobytes() == op.find_all(f).tobytes(), i
    with pytest.raises(api.UgxError):
        sc.fetch(n, 1)


def test_overflow_and_bad_arguments(api):
    sc = api.Scanner(0)
    pat = api.Pattern.load(cfg("c5"), 0)
    op = LO.oracle(cfg("c5"))
    files = make_files("c5", np.random.default_rng(13), 20)
    buf, begins, lens = pack(files)
    for lines in (False, True):
        dt = api.LINE_DTYPE if lines else api.MATCH_DTYPE
        rc, n, first, t, _ = raw(api, sc, pat, buf, begins, lens, lines)
        assert rc == 0 and n > 1 and t.matches == n
        # too small: UGX_E_OVERFLOW, *n_out and first[] filled, the records still fetchable
        rc, n2, first2, _, _ = raw(api, sc, pat, buf, begins, lens, lines, cap=n - 1, out=np.zeros(n, dtype=dt))
        assert rc == 5 and n2 == n and (first2 == first).all()
        got = sc.fetch_lines(0, n) if lines else sc.fetch(0, n)
        for i, f in enumerate(files):
            want = op.find_lines(f) if lines else op.find_all(f)
            assert got[int(first[i]):int(first[i + 1])].tobytes() == want.tobytes(), (lines, i)
        rc, n3, _, _, out = raw(api, sc, pat, buf, begins, lens, lines, cap=n, out=np.zeros(n, dtype=dt))
        assert rc == 0 and n3 == n and out.tobytes() == got.tobytes()
        # a misaligned begin, a file past the buffer end, a NULL first[]
        bad = begins.copy()
        bad[3] += 1
        assert raw(api, sc, pat, buf, bad, lens, lines)[0] == 1
        long_ = lens.copy()
        long_[-1] = buf.size
        assert raw(api, sc, pat, buf, begins, long_, lines)[0] == 1
        assert raw(api, sc, pat, buf, begins, lens, lines, first=False)[0] == 1
        # no files: UGX_OK, first[0] = 0, no records
        rc, n, first, t, _ = raw(api, sc, pat, buf, begins, lens, lines, nfiles=0)
        assert rc == 0 and n == 0 and int(first[0]) == 0 and t.matches == 0
    # unknown flags
    assert raw(api, sc, pat, buf, begins, lens, True, flags=2)[0] == 1
    assert b"unknown flags" in api.lib().ugx_last_error()
    # the Python forms of an empty batch and of empty files
    rec, first, tot = sc.find_lines_batch(pat, [])
    assert len(rec) == 0 and list(first) == [0]
    rec, first, tot = sc.find_all_batch(pat, [b"", b""])
    assert len(rec) == 0 and list(first) == [0, 0, 0]
