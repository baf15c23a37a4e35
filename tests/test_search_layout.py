"""CPU model of count_lines_search_kernel's work layout (csrc/stream_search.cu), on the automaton that
ugx_search_describe returns: a 16 KiB region is cut into lane stretches of S bytes; each stretch runs the automaton
from the empty set D - 1 bytes before its start and carries its state across its 32-byte steps; each lane resolves
its lines per step on its own (stretch_step); per group of 32 stretches the warp chains the lanes with the three
ballots and the carry add (combine_stretches); the region summaries are chained as in stream_epilogue.  The count
must be the oracle's `ugrep -c` count, for stretch lengths around the kernel's and with lines, matches and newlines
across stretch and region edges."""
import os

import numpy as np
import pytest

import golden_lib as G
import oracle_lib as O
import test_search_dfa as T
from ugrep_b200 import corpus

REGION = 16384
STEP = 32
M32 = np.uint64(0xFFFFFFFF)
PAT_DIR = os.path.join(O.ROOT, "ugrep_b200", "patterns")


def _popc(x):
    return np.bitwise_count(x).astype(np.int64)


def stretch_flags(info, cls, table, a, S):
    """per stretch (in address order): the flag word of stretch_step (bit 0 newline, bit 1 head success, bit 2 open
    success) and the lane-private count; bytes past the end read as 0 and never succeed"""
    n = a.size
    npad = -(-n // REGION) * REGION
    buf = np.zeros(npad, dtype=np.uint8)
    buf[:n] = a
    starts = np.arange(0, npad, S, dtype=np.int64)
    st = np.full(starts.size, info.classes, dtype=np.int64)
    for j in range(info.depth - 1, 0, -1):                       # warm-up; '\n' before the buffer's start
        p = starts - j
        st = table[st + cls[np.where(p >= 0, buf[np.maximum(p, 0)], 10)]]
    f = np.zeros(starts.size, dtype=np.uint64)
    lcount = 0
    one = np.uint64(1)
    for s0 in range(0, S, STEP):
        succ = np.zeros(starts.size, dtype=np.uint64)
        nl = np.zeros(starts.size, dtype=np.uint64)
        for k in range(STEP):
            p = starts + s0 + k
            b = buf[p]
            st = table[st + cls[b]]
            succ |= ((st == 0) & (p < n)).astype(np.uint64) << np.uint64(k)
            nl |= (b == 10).astype(np.uint64) << np.uint64(k)
        # stretch_step
        s = succ & ~nl & M32
        total = s + (~nl & M32)
        g = (total >> np.uint64(32)) & one
        v = total & M32 & nl
        first = nl & ((~nl + one) & M32)
        has = (nl != 0).astype(np.uint64)
        hs = np.where(has == 1, ((v & first) != 0).astype(np.uint64), g)
        tnl, topen = f & one, (f >> np.uint64(2)) & one
        lcount += int((tnl & hs & (topen ^ one)).sum()) + int(np.where(has == 1, _popc(v & ~first & M32) + g.astype(np.int64), 0).sum())
        head = ((f >> one) & one) | ((tnl ^ one) & hs)
        opn = np.where(has == 1, g, topen | hs)
        f = (tnl | has) | (head << one) | (opn << np.uint64(2))
    return f, lcount


def layout_count(info, cls, table, a, S):
    f, lcount = stretch_flags(info, cls, table, a, S)
    per_region = REGION // S
    ucount = 0
    sums = []
    for r in range(f.size // per_region):
        cin, seen, head = 1, False, False
        for h in range(0, per_region, 32):                       # combine_stretches, groups of 32 lanes in order
            lanes = [int(x) for x in f[r * per_region + h:r * per_region + h + 32]]
            lanes += [0] * (32 - len(lanes))
            NL = sum(((x & 1) << l) for l, x in enumerate(lanes))
            H = sum((((x >> 1) & 1) << l) for l, x in enumerate(lanes))
            Gb = sum((((x >> 2) & 1) << l) for l, x in enumerate(lanes))
            A = (Gb | ~NL) & 0xFFFFFFFF
            carry = A + Gb + cin
            C = (carry ^ A ^ Gb) & 0xFFFFFFFF
            if not seen:
                headlanes = ((NL & -NL) << 1) - 1 if NL else 0xFFFFFFFF
                if H & headlanes:
                    head = True
            ucount += bin(H & ~C & 0xFFFFFFFF).count("1")
            cin = carry >> 32
            if NL:
                seen = True
        sums.append((seen, head, cin if seen else int(head)))
    adjust, c = 0, 0                                             # stream_epilogue: chain the region summaries
    for nl, hd, g in sums:
        if hd and not c:
            adjust += 1
        c = g if nl else (c | int(hd))
    return lcount + ucount + adjust


def _eligible_golden():
    return [n for n in G.pattern_names() if T.describe(G.pattern_path(n))[0].eligible]


@pytest.mark.parametrize("S", [256, 128, 512])
@pytest.mark.parametrize("name", _eligible_golden())
def test_golden_cases_across_stretch_and_region_edges(name, S):
    path = G.pattern_path(name)
    info, cls, table = T.describe(path)
    op = O.OraclePattern(path)
    filler = np.frombuffer((b"#" * 63 + b"\n") * 512, dtype=np.uint8)
    rng = np.random.default_rng(len(name) * 1000 + S)
    for _, data in G.cases(name):
        d = np.frombuffer(data, dtype=np.uint8)[:4096]
        nl = np.frombuffer(b"\n", dtype=np.uint8)
        # the case's first byte at, and a few bytes around, a stretch edge and a region edge, and at a random offset
        for off in [S - 1, S, S + 3, 2 * S - 9, REGION - 5, REGION + 1] + [int(x) for x in rng.integers(0, 2 * S, 2)]:
            buf = np.concatenate([filler[:off], nl, d, nl, filler[:S + 7]])
            assert layout_count(info, cls, table, buf, S) == op.count_lines(buf.tobytes()), (off, S)


@pytest.mark.parametrize("S", [256, 128, 512])
@pytest.mark.parametrize("cname", ["c2", "c2s", "c4"])
def test_config_blocks(cname, S):
    path = os.path.join(PAT_DIR, ("c4" if cname == "c4" else "c2") + ".ugxp")
    info, cls, table = T.describe(path)
    op = O.OraclePattern(path)
    blk = corpus.block(cname, 1 << 20)
    for cut in (0, 5, S // 2 + 3):
        a = blk[cut:]
        assert layout_count(info, cls, table, a, S) == op.count_lines(a.tobytes()), (cut, S)


def test_long_lines_and_matches_across_stretch_edges():
    info, cls, table = T.describe(os.path.join(PAT_DIR, "c2.ugxp"))
    op = O.OraclePattern(os.path.join(PAT_DIR, "c2.ugxp"))
    word = np.frombuffer(corpus.words_list()[7], dtype=np.uint8)
    for S in (128, 256, 512):
        a = np.full(3 * REGION + 300, ord("#"), dtype=np.uint8)
        # a match that starts in the warm-up bytes of a stretch and decides inside it, one at every region edge, a
        # line longer than a region with a match only in its last stretch, and lines that end on stretch edges
        for at in (S - 3, 5 * S - len(word) // 2, REGION - 2, 2 * REGION - len(word) + 1, 3 * REGION + 100):
            a[at:at + len(word)] = word
        for at in (2 * S - 1, 7 * S, REGION + S, 3 * REGION + 50):
            a[at] = 10
        assert layout_count(info, cls, table, a, S) == op.count_lines(a.tobytes()), S
