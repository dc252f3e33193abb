"""Lines without a GPU: the numpy reference of a record's line position, and sharding.line_origins (the
host half of line positions over shards) against it."""
import random

import numpy as np
import pytest

from omega_match_b200.sharding import NO_NEWLINE, line_origins


def positions(hay: np.ndarray, offsets: np.ndarray) -> np.ndarray:
    """(line, begin, end) per offset (include/olm_b200.h "lines"): '\\n' count before it, one past the
    last '\\n' before it (or 0), the first '\\n' at or after it (or the size)."""
    hay = np.asarray(hay, dtype=np.uint8)
    nl = np.flatnonzero(hay == 10).astype(np.int64)
    i = np.searchsorted(nl, np.asarray(offsets, dtype=np.int64), side="left")
    pad = np.concatenate([[-1], nl, [hay.size]])  # pad[i] = the '\n' before, pad[i + 1] = the one at or after
    out = np.zeros((i.size, 3), dtype=np.uint64)
    out[:, 0], out[:, 1], out[:, 2] = i, pad[i] + 1, pad[i + 1]
    return out


def facts(hay: np.ndarray, b: int, e: int):
    nl = np.flatnonzero(hay[b:e] == 10)
    return (int(nl.size), int(nl[0]) if nl.size else None, int(nl[-1]) if nl.size else None)


def test_reference_on_hand_made_haystacks():
    hay = np.frombuffer(b"ab\ncd\r\n\nx\ry", dtype=np.uint8)
    got = positions(hay, np.arange(hay.size))
    want = [(0, 0, 2), (0, 0, 2), (0, 0, 2), (1, 3, 6), (1, 3, 6), (1, 3, 6), (1, 3, 6), (2, 7, 7),
            (3, 8, 11), (3, 8, 11), (3, 8, 11)]
    assert got.tolist() == [list(w) for w in want]
    assert positions(np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.int64)).shape == (0, 3)
    assert positions(np.frombuffer(b"abc", dtype=np.uint8), [0, 2]).tolist() == [[0, 0, 3], [0, 0, 3]]
    assert positions(np.frombuffer(b"\n\n", dtype=np.uint8), [0, 1]).tolist() == [[0, 0, 0], [1, 1, 1]]


@pytest.mark.parametrize("seed", range(40))
def test_line_origins_against_the_reference(seed):
    rng = random.Random(seed)
    n = rng.choice([0, 1, 7, 100, 1000, 5000])
    density = rng.choice([0.0, 0.001, 0.05, 0.5, 1.0])
    hay = np.where(np.random.default_rng(seed).random(n) < density, 10, 97).astype(np.uint8)
    k = rng.randint(1, 8)
    cuts = sorted(rng.randint(0, n) for _ in range(k - 1))
    edges = [0] + cuts + [n]  # (equal cuts: empty ranges)
    ranges = list(zip(edges[:-1], edges[1:]))
    f = [facts(hay, b, e) for b, e in ranges]
    origins = line_origins(f, ranges, n)
    whole = positions(hay, np.arange(n))
    for (b, e), (line, begin, nxt) in zip(ranges, origins):
        # what a shard computes from its own bytes and its origin equals the whole-haystack answer
        own = hay[b:e]
        nl = np.flatnonzero(own == 10)
        for o in range(b, e):
            p = o - b
            i = int(np.searchsorted(nl, p))
            want = whole[o].tolist()
            got = [line + i, b + int(nl[i - 1]) + 1 if i else begin, b + int(nl[i]) if i < nl.size else nxt]
            assert got == want, (seed, ranges, o)
        if b < n:
            assert [line, begin] == whole[b].tolist()[:2]
        nl_after = np.flatnonzero(hay[e:] == 10)
        assert nxt == (e + int(nl_after[0]) if nl_after.size else n)


def test_line_origins_accepts_the_library_none_and_checks_ranges():
    f = [(0, NO_NEWLINE, NO_NEWLINE), (1, 2, 2)]
    assert line_origins(f, [(0, 4), (4, 8)], 8) == [(0, 0, 6), (0, 0, 8)]
    with pytest.raises(ValueError):
        line_origins(f, [(0, 4), (5, 8)], 8)
    with pytest.raises(ValueError):
        line_origins(f, [(0, 4), (4, 8)], 9)
    with pytest.raises(ValueError):
        line_origins(f[:1], [(0, 4), (4, 8)], 8)
