"""`-c` through count_lines_search_kernel (csrc/stream_search.cu) against the same call with the scanner option
"no_search" (count_lines_stream_kernel alone) and against the oracle: matches placed across lane segments (64 bytes),
blocks (2 KiB), regions (16 KiB) and the end of the buffer, where the candidate test applies again; long lines, a buffer
without a newline, lengths around region multiples, host / pinned / device / misaligned buffers, newline counting,
the sharded form and the reported kernel."""
import os

import numpy as np
import pytest

import golden_lib as G
import oracle_lib as O
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu

PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")
C2 = os.path.join(PAT_DIR, "c2.ugxp")


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api
    return api


@pytest.fixture(scope="module")
def scanners(api):
    """(search route, today's route); both take the streaming kernels for every eligible DFA pattern"""
    a, b = api.Scanner(0), api.Scanner(0)
    for s in (a, b):
        s.set_option("stream_dfa", 1)
    b.set_option("no_search", 1)
    return a, b


def _eligible_golden():
    import test_search_dfa as T
    return [n for n in G.pattern_names() if T.describe(G.pattern_path(n))[0].eligible]


def check(scanners, pat, op, data, want=None):
    a, b = scanners
    want = op.count_lines(data) if want is None else want
    ta, tb = a.count_lines(pat, data), b.count_lines(pat, data)
    assert ta.matches == want and tb.matches == want, (ta.matches, tb.matches, want)
    return ta, tb


@pytest.mark.parametrize("name", _eligible_golden())
def test_golden_cases_across_segment_block_and_region_edges(api, scanners, name):
    import torch
    path = G.pattern_path(name)
    pat = api.Pattern.load(path, 0)
    op = O.OraclePattern(path)
    filler = np.frombuffer((b"#" * 63 + b"\n") * 1024, dtype=np.uint8)   # 64 KiB of lines no pattern here matches
    for case, data in G.cases(name):
        d = np.frombuffer(data, dtype=np.uint8)
        if d.size > 8192:
            d = d[:8192]
        for off in list(range(0, 64)) + [2048 - 5, 2048 + 3, 16384 - 9, 16384 - 1, 16384, 32768 - 7]:
            buf = np.concatenate([filler[:off], np.frombuffer(b"\n", dtype=np.uint8), d,
                                  np.frombuffer(b"\n", dtype=np.uint8), filler])
            dev = torch.from_numpy(buf).cuda()
            check(scanners, pat, op, dev, op.count_lines(buf.tobytes()))
        # the same text as the last bytes of the buffer, where positions also need the candidate test
        for tail in (0, 1, 7, 23, 24, 25, 535, 536, 600, 16384 + 30):
            buf = np.concatenate([filler, filler[:tail], d])
            check(scanners, pat, op, torch.from_numpy(buf).cuda(), op.count_lines(buf.tobytes()))


def test_lengths_around_region_multiples(api, scanners):
    import torch
    pat = api.Pattern.load(C2, 0)
    op = O.OraclePattern(C2)
    blk = corpus.block("c2", 1 << 20)
    for k in (1, 2, 5, 33):
        for extra in (0, 1, 15, 16, 535, 536, 537):
            n = k * 16384 + extra
            data = np.resize(blk, n)
            ta, _ = check(scanners, pat, op, torch.from_numpy(data).cuda(), op.count_lines(data.tobytes()))
            assert ta.kernel == "count_lines_search_kernel"


def test_long_lines_and_no_newline(api, scanners):
    import torch
    pat = api.Pattern.load(C2, 0)
    op = O.OraclePattern(C2)
    word = corpus.words_list()[7]
    n = 256 << 20
    line = torch.full((n,), ord("#"), dtype=torch.uint8, device="cuda")
    check(scanners, pat, op, line, 0)                                            # no newline, no match
    w = torch.tensor(list(word), dtype=torch.uint8, device="cuda")
    line[n // 2 + 5:n // 2 + 5 + len(word)] = w
    check(scanners, pat, op, line, 1)                                            # no newline, one match mid-line
    line[-1] = 10
    check(scanners, pat, op, line, 1)                                            # one 256 MiB line with a match
    line[n // 2 + 5:n // 2 + 5 + len(word)] = ord("#")
    line[n - 1 - len(word):n - 1] = w
    check(scanners, pat, op, line, 1)                                            # ... the match at its very end
    line[n - 1 - len(word):n - 1] = ord("#")
    check(scanners, pat, op, line, 0)                                            # ... and without one
    # lines longer than a region, a match across each region edge
    blk = np.full(5 * 16384, ord("#"), dtype=np.uint8)
    for r in range(1, 5):
        blk[r * 16384 - 3:r * 16384 - 3 + len(word)] = np.frombuffer(word, dtype=np.uint8)
    blk[2 * 16384 + 100] = 10
    check(scanners, pat, op, torch.from_numpy(blk).cuda(), op.count_lines(blk.tobytes()))


def test_host_pinned_device_misaligned_and_newlines(api, scanners):
    import torch
    a, b = scanners
    pat = api.Pattern.load(C2, 0)
    op = O.OraclePattern(C2)
    for cname in ("c2", "c2s"):
        blk = corpus.block(cname, 96 << 20)   # >= two pipeline chunks: the host buffers take the overlapped copy
        want = op.count_lines(blk)
        for src in (blk, torch.from_numpy(blk.copy()).pin_memory().numpy(), torch.from_numpy(blk).cuda()):
            ta, tb = check(scanners, pat, op, src, want)
            assert ta.kernel == "count_lines_search_kernel" and tb.kernel == "count_lines_stream_kernel"
        dev = torch.from_numpy(blk).cuda()
        for cut in (1, 3, 17):
            check(scanners, pat, op, dev[cut:], op.count_lines(blk[cut:]))
        a.set_option("count_newlines", 1)
        t = a.count_lines(pat, dev)
        a.set_option("count_newlines", 0)
        assert t.matches == want and t.flags & 1 and t.newlines == int((blk == 10).sum())


def test_full_size_by_additivity(api, scanners):
    import torch
    a, _ = scanners
    for cname, gib in (("c2", 4), ("c2s", 4), ("c4", 8)):
        path = os.path.join(PAT_DIR, ("c4" if cname == "c4" else "c2") + ".ugxp")
        pat = api.Pattern.load(path, 0)
        block = corpus.block(cname, 32 << 20)
        reps = int(gib * (1 << 30)) // len(block)
        dev = torch.from_numpy(block).cuda().repeat(reps)
        t = a.count_lines(pat, dev)
        assert t.matches == reps * O.OraclePattern(path).count_lines(block), cname
        assert t.kernel == "count_lines_search_kernel" and t.launches == 1
        del dev


def test_sharded_form(api):
    blk = corpus.block("c2", 80 << 20)
    want = O.OraclePattern(C2).count_lines(blk)
    sh = api.Sharded(C2, [0])
    tot, _, _ = sh.scan(blk, "lines")
    sh.set_option("no_search", 1)
    tot2, _, _ = sh.scan(blk, "lines")
    assert tot.matches == want and tot2.matches == want


def test_kernel_per_route(api):
    import torch
    blk = torch.from_numpy(corpus.block("c2", 4 << 20)).cuda()
    pat = api.Pattern.load(C2, 0)
    sc = api.Scanner(0)
    assert sc.count_lines(pat, blk).kernel == "count_lines_search_kernel"
    sc.set_option("no_search", 1)
    assert sc.count_lines(pat, blk).kernel == "count_lines_stream_kernel"
    sc.set_option("no_search", 0)
    c1 = api.Pattern.load(os.path.join(PAT_DIR, "c1.ugxp"), 0)
    assert sc.count_lines(c1, torch.from_numpy(corpus.block("c1", 4 << 20)).cuda()).kernel == "count_lines_literal_kernel"
