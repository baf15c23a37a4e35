"""count_lines_search_kernel's lane stretches on the device (csrc/stream_search.cu): the default route against the
scanner option "no_search" (count_lines_stream_kernel) and the oracle, with matches and newlines at every offset of a
stretch on both sides of lane-stretch edges, of the edge between a round's two halves (the lane's second chain) and
of region edges, in interior regions and in the region at the end of the buffer; buffers of 1, 2, 3, 5 and 7 regions
and more; lines longer than a stretch and than a region; newline counting; a device buffer at 16 mod 32."""
import os

import numpy as np
import pytest

import oracle_lib as O
from ugrep_b200 import corpus

pytestmark = pytest.mark.gpu

PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")
C2 = os.path.join(PAT_DIR, "c2.ugxp")
REGION = 16384
S = 256          # bytes per lane stretch (UGX_SEARCH_S); the sweep below also crosses every edge of 128-byte stretches
HALF = 32 * S    # the second chain of a lane starts here in each region


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests must run on the B200 box")
    from ugrep_b200 import api
    return api


@pytest.fixture(scope="module")
def scanners(api):
    a, b = api.Scanner(0), api.Scanner(0)
    b.set_option("no_search", 1)
    return a, b


def check(scanners, pat, op, data, newlines=False):
    import torch
    a, b = scanners
    want = op.count_lines(data.tobytes())
    dev = torch.from_numpy(data).cuda()
    ta, tb = a.count_lines(pat, dev), b.count_lines(pat, dev)
    assert ta.kernel == "count_lines_search_kernel"
    assert ta.matches == want and tb.matches == want, (ta.matches, tb.matches, want)
    if newlines:
        a.set_option("count_newlines", 1)
        t = a.count_lines(pat, dev)
        a.set_option("count_newlines", 0)
        assert t.matches == want and t.newlines == int((data == 10).sum())


def test_every_offset_around_stretch_half_and_region_edges(api, scanners):
    pat, op = api.Pattern.load(C2, 0), O.OraclePattern(C2)
    word = np.frombuffer(max(corpus.words_list(), key=len), dtype=np.uint8)   # the longest needle: its decision
    n = 3 * REGION + 3000                                                     # spans the most warm-up bytes
    # lane-stretch edges, the second chain's first stretch, region edges; regions 0-2 interior, region 3 at the end
    edges = [S, 2 * S, 31 * S, HALF, HALF + S, REGION, REGION + HALF, 2 * REGION + 3 * S, 3 * REGION, 3 * REGION + 2 * S]
    for k in range(S):
        a = np.full(n, ord("#"), dtype=np.uint8)
        for i, e in enumerate(edges):
            a[e - S + k:e - S + k + word.size] = word[:max(0, min(word.size, n - (e - S + k)))]
            if i % 3 != 1:                   # some edges keep no newline: those lines span two edges
                a[e - S + (k + S // 2 + 7 * i) % S] = 10
        check(scanners, pat, op, a, newlines=k % 16 == 0)


def test_region_counts(api, scanners):
    for cname, pname in (("c2", "c2"), ("c2s", "c2"), ("c4", "c4")):
        path = os.path.join(PAT_DIR, pname + ".ugxp")
        pat, op = api.Pattern.load(path, 0), O.OraclePattern(path)
        blk = corpus.block(cname, 1 << 20)
        for k in (1, 2, 3, 5, 7, 64):
            for extra in (0, 17, 3000):
                check(scanners, pat, op, np.resize(blk, k * REGION + extra), newlines=extra == 17)


def test_lines_longer_than_a_stretch_and_a_region(api, scanners):
    pat, op = api.Pattern.load(C2, 0), O.OraclePattern(C2)
    word = np.frombuffer(corpus.words_list()[3], dtype=np.uint8)
    n = 6 * REGION + 1000
    for at in (S - 2, HALF - 1, HALF + 5 * S + 3, REGION - 4, 3 * REGION + HALF - 2, 5 * REGION + 17):
        for nl in ((), (at - 2 * S,), (at + S + 1,), (at - REGION - 3, at + REGION + 3)):
            a = np.full(n, ord("#"), dtype=np.uint8)
            a[at:at + word.size] = word
            for p in nl:
                if 0 <= p < n:
                    a[p] = 10
            check(scanners, pat, op, a)


def test_device_buffer_at_16_mod_32(api, scanners):
    """a 16-byte aligned device buffer is scanned in place; at 16 mod 32 the steps take two 16-byte loads"""
    import torch
    a, b = scanners
    pat, op = api.Pattern.load(C2, 0), O.OraclePattern(C2)
    data = np.resize(corpus.block("c2", 1 << 20), 7 * REGION + 3000)
    dev = torch.from_numpy(np.concatenate([np.zeros(16, dtype=np.uint8), data])).cuda()[16:]
    assert dev.data_ptr() % 32 == 16
    want = op.count_lines(data.tobytes())
    assert a.count_lines(pat, dev).matches == want and b.count_lines(pat, dev).matches == want
