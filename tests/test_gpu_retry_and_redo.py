"""The two places where the scan gives work a second try, against the oracle -- needs a B200 (the
oracle companion of the retry shapes runs without one).

* The retried call (engine.cu match_device): a fresh engine sizes its result buffer for
  max(out_hint, n/64 + 4096) records; a call with more records than that runs its whole launch
  sequence again with a buffer of the exact size.  Every retried call here is the first call of a
  matcher, and asserts on the oracle that its record count is above that first capacity.
* The redone chunk (scan.cu redo_kernel): a 512-byte chunk whose matches do not fit its staging
  area -- at most kChunkCapMax = 1024 entries in any geometry -- is only counted by the scan and
  then built again and written directly; so is a record whose source length needs 23 bits or more.
  The dense regions below put more than 1024 matches into single chunks.

Calls on one matcher are replayed in the same order on one oracle: under word_boundary the image of
the reference's scratch buffer that earlier calls left behind decides matches (SURVEY H6).
"""
import ctypes as C
import functools
import os

import numpy as np
import pytest

import inputs
from conftest import describe_diff, same_matches
from omega_match_b200 import Matcher, _lib
from oracle.oracle import Oracle

W = inputs.WINDOW
TILE = 4096           # scan.cuh OLM_TILE_BYTES
CHUNK = 512           # scan.cuh kChunkBytes
CHUNK_CAP_MAX = 1024  # scan.cuh kChunkCapMax: no staging area holds more matches of one chunk


def first_capacity(n: int) -> int:
    """Records a fresh engine makes room for in a call over n bytes (engine.cu match_device)."""
    return n // 64 + 4096


def check(m: Matcher, o: Oracle, hay, **flags):
    got = m.match_arrays(hay, **flags)
    want = o.match(hay, **flags)
    assert same_matches(got, want), f"{flags}: " + describe_diff(got, want)
    return want


def check_retried(m: Matcher, o: Oracle, hay, **flags):
    """check() of the first call of a fresh matcher that has more records than its first capacity."""
    want = check(m, o, hay, **flags)
    assert want.size > first_capacity(len(hay)), (want.size, first_capacity(len(hay)))
    return want


def _stats(m: Matcher):
    st = m.get_match_stats()
    return st.total_hits, st.total_misses, st.total_filtered, st.total_attempts, st.total_comparisons


def _oracle_stats(o: Oracle):
    ref = o.stats.as_dict()
    return ref["hits"], ref["misses"], ref["filtered"], ref["attempts"], ref["comparisons"]


def store_info(path) -> dict:
    info = _lib.StoreInfoC()
    assert _lib.load().olm_store_inspect(os.fsencode(path), C.byref(info)) == 0
    return info.as_dict()


@functools.lru_cache(maxsize=4)
def tiled_text(n: int, seed: int) -> bytes:
    """n bytes of text_haystack: a 1 MiB + 7 piece repeated (long haystacks without a long wait)."""
    piece = inputs.text_haystack((1 << 20) + 7, seed).tobytes()
    return (piece * (n // len(piece) + 1))[:n]


# ---- 1. a retry starts from the image of the scratch buffer the call started with -------------------
#
# A store that drops bytes (ignore-punctuation or elide-whitespace) with 2..4 byte patterns, called
# with word_boundary, reads the stale tail of each window from the image of the scratch buffer and then
# writes the call's windows into it (transform.cu window_descs_launch).  A window whose tail comes from
# the image, at an index M_w that a later window of the same call writes, is where a retry that reads
# the image its own first attempt left behind goes wrong.

SHORT_PATS = b"ab\nzq\nhello\n"


def dense_ab(n: int) -> bytes:
    """n bytes of "ab ab ab ...": one record per 3 bytes, with word_boundary too."""
    return (b"ab " * (n // 3 + 1))[:n]


def two_window_hay() -> bytes:
    """Window 0 normalises to " ab" (M_0 = 3, no trim: its tail is image byte 3); window 1 writes
    "ab ab ..." there -- a 'b' that turns the match at the end of window 0 into no match."""
    return b"." * (W - 3) + b" ab" + dense_ab(W // 2)


def three_window_hay() -> bytes:
    """Window 1 normalises to 1000 bytes ending in " ab": its tail is image byte 1000, since window 0
    (" hello", extent 6) does not reach it; window 2 ("ab ab ...", extent > 1000) writes it.  Window 0
    ends in a 5-byte pattern, whose end never reads a stale tail."""
    return b"." * (W - 6) + b" hello" + b"." * (W - 1000) + b"x" * 997 + b" ab" + dense_ab(W // 2)


def span_hay() -> bytes:
    """two_window_hay with a full window 1 and a third window: in 8 MiB spans the first span is the
    two-window shape."""
    return b"." * (W - 3) + b" ab" + dense_ab(W) + b"zq ." * 300


SHAPES = {"two-windows": (two_window_hay, (0, 1, 0)), "two-windows-elide": (two_window_hay, (0, 1, 1)),
          "three-windows": (three_window_hay, (0, 1, 0)), "spans": (span_hay, (0, 1, 0))}


def _fresh(sf) -> Oracle:
    return Oracle.from_patterns(SHORT_PATS, *map(bool, sf))


@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_retry_shapes_depend_on_the_image(shape):
    """Each shape answers differently from a fresh image and from the image its own call leaves
    behind -- what a first attempt leaves to a second one; so a retry that reads the latter is caught."""
    make, sf = SHAPES[shape]
    hay = make()
    fresh = _fresh(sf).match(hay, word_boundary=True)
    advanced = _fresh(sf)
    advanced.match(hay, word_boundary=True)
    again = advanced.match(hay, word_boundary=True)
    assert not same_matches(fresh, again), shape
    if shape == "two-windows":
        assert (fresh.size, again.size) == (699_052, 699_051)
        assert (W - 2, 2) in set(zip(fresh["offset"].tolist(), fresh["len"].tolist()))
    assert fresh.size > first_capacity(len(hay))


def _image_dependent(sf, first_hay, first_flags, shorts):
    """The short word_boundary calls whose answer after a call over `first_hay` differs from a fresh
    matcher's."""
    out = []
    for s in shorts:
        after = _fresh(sf)
        after.match(first_hay, **first_flags)
        if not same_matches(after.match(s, word_boundary=True), _fresh(sf).match(s, word_boundary=True)):
            out.append(s)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["two-windows", "two-windows-elide", "three-windows"])
def test_retried_call_reads_the_image_it_started_with(store_cache, shape):
    make, sf = SHAPES[shape]
    path = store_cache("retry-short", SHORT_PATS, sf)
    hay = make()
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        check_retried(m, o, hay, word_boundary=True)
        # and leaves the oracle's image behind
        for short in (b"x ab", b"xyzw.ab", b"." * 9 + b"q ab"):
            check(m, o, short, word_boundary=True)


@pytest.mark.gpu
@pytest.mark.parametrize("sf,flags", [((1, 0, 0), {"word_boundary": True}), ((0, 1, 1), {})])
def test_retried_calls_that_keep_the_image_elsewhere(store_cache, sf, flags):
    """Case folding only (the window descriptors read image bytes no window of the call writes) and a
    normalising store without word_boundary (the image is brought up to date after the scan, the same
    way in every attempt): the retried call, then short calls whose answer depends on the image."""
    path = store_cache("retry-short", SHORT_PATS, sf)
    hay = two_window_hay()
    shorts = [b"x ab", b"ab", b"q.ab", b"xyzw ab", b"." * 9 + b"q ab", b"x" * 1000 + b" ab"]
    dependent = _image_dependent(sf, hay, flags, shorts)
    assert dependent, "no short call depends on the image"
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        check_retried(m, o, hay, **flags)
        for short in dependent:
            check(m, o, short, word_boundary=True)


@pytest.mark.gpu
def test_retried_call_of_two_launch_groups(store_cache):
    """65 windows: two launch groups, the second carrying the total of the first, retried, under
    word_boundary.  Window 0 reads its tail from the image (M_0 = 3) and the last window writes it; dense
    regions ("a a a ...": every "a" starts 8 patterns) lie in both groups."""
    pats = SHORT_PATS + b"\n".join(b" ".join([b"a"] * k) for k in range(1, 9)) + b"\nthe\nand\nof\n"
    path = store_cache("retry-groups", pats, (0, 1, 0))
    n = (257 << 20) + 12345
    hay = bytearray(tiled_text(n, 41))
    hay[:W] = b"." * (W - 3) + b" ab"
    hay[10 * W:10 * W + (256 << 10)] = (b" " + b"a " * (128 << 10))[:256 << 10]
    last = 64 * W
    hay[last:] = (b"zzzz " + b"a " * ((n - last) // 2))[:n - last]
    hay = bytes(hay)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        check_retried(m, o, hay, word_boundary=True)
        check(m, o, b"x ab", word_boundary=True)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["plain", "normalising"])
def test_retried_call_counts_statistics_once(store_cache, kind):
    """Exact statistics (all five counters) of a retried call equal the oracle's: a second attempt
    counts from zero."""
    if kind == "plain":
        pats = b"\n".join([b"a" * k for k in range(1, 13)] + [b"the", b"shall"])
        path = store_cache("retry-stats-plain", pats)
        hay = inputs.text_haystack(300_000, 3).tobytes() + b"a" * 30_000 + b" the end"
        calls = [{}, {"longest_only": True}]
    else:
        path = store_cache("retry-short", SHORT_PATS, (0, 1, 0))
        hay = two_window_hay()
        calls = [{"word_boundary": True}]
    for flags in calls:
        o = Oracle.from_olm(path)
        with Matcher(path) as m:
            m.set_exact_stats(True)
            check_retried(m, o, hay, **flags)
            assert _stats(m) == _oracle_stats(o), flags


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["pattern_counts", "match_ids", "host-spans", "stream", "two-engines"])
def test_retried_call_through_every_entry_point(store_cache, monkeypatch, entry):
    """The two-window shape through the other entry points that end in a device call: pattern counts,
    pattern ids, OLM_HOST_SPAN_BYTES spans (8 MiB: the first span is the two-window shape), one stream
    push, and a matcher of two engines (under word_boundary the call goes to the first one alone)."""
    from test_gpu_multi import _devices
    from test_gpu_pattern_counts import _oracle_counts
    from test_gpu_pattern_ids import _check_ids
    sf = (0, 1, 0)
    path = store_cache("retry-short", SHORT_PATS, sf)
    o = Oracle.from_olm(path)
    hay = two_window_hay()
    if entry == "host-spans":
        monkeypatch.setenv("OLM_HOST_SPAN_BYTES", str(2 * W))
        hay = span_hay()
    with Matcher(path, devices=_devices(2) if entry == "two-engines" else None) as m:
        if entry == "pattern_counts":
            want, n = _oracle_counts(m, o, hay, sf, word_boundary=True)
            assert n > first_capacity(len(hay))
            got = m.pattern_counts(hay, word_boundary=True)
            assert (got == want).all(), (got, want)
        elif entry == "match_ids":
            m.set_pattern_ids(True)
            got = m.match_ids(hay, word_boundary=True)
            want = o.match(hay, word_boundary=True)
            assert same_matches(got, want), describe_diff(got, want)
            assert want.size > first_capacity(len(hay))
            _check_ids(m, hay, got, sf, "retried")
            m.set_pattern_ids(False)
        elif entry == "stream":
            with m.stream(word_boundary=True) as s:
                got = s.push(hay, last=True)
            want = o.match(hay, word_boundary=True)
            assert same_matches(got, want), describe_diff(got, want)
            assert want.size > first_capacity(len(hay))
        else:
            check_retried(m, o, hay, word_boundary=True)
        check(m, o, b"x ab", word_boundary=True)


# ---- 2. redone chunks on every variant of the scan kernel ---------------------------------------------
#
# Each store kind selects one filter layout of scan_kernel (G: key filter, Q: 1..3 byte candidates,
# C: byte-class prefilter, SX: second look at short candidates, COOP: warp-cooperative compare); a store
# flag adds XF (the chunks are transformed on chip).  Exact statistics select the generic path
# (FAST = 0), whose counters must not count a redone chunk twice.
#
# Two dense units: a run of one byte (every position starts several patterns: dense without a start or
# end predicate) and short words (every word starts several patterns made of words joined by spaces:
# dense under word_boundary and word_suffix too).  longest_only keeps one match per position and a line
# predicate one per line: such calls overflow only the staging areas smaller than kChunkCapMax.

DENSE_FLAGSETS = [{}, {"longest_only": True}, {"longest_only": True, "no_overlap": True}, {"word_boundary": True},
                  {"line_start": True, "line_end": True}, {"word_suffix": True}]
SPARSE = [b"shall", b"unto", b"people", b"king"]
AA_WORDS = [b" ".join([b"aa"] * k) for k in range(2, 10)]  # 8 patterns start at every "aa " word


def _coop_patterns(with_short: bool) -> list:
    """4-byte keys with 4, 31, 32, 33 and 400 records behind them; of the 400, 40 are prefixes of each
    other (a position in a run of x has up to 41 matches) and 360 are not."""
    pats = [b"bbbb" + b"b" * j for j in range(1, 5)] + [b"cccc" + b"c" * j for j in range(1, 32)]
    pats += [b"dddd" + b"d" * j for j in range(1, 33)] + [b"eeee" + b"e" * j for j in range(1, 34)]
    pats += [b"xxxx" + b"x" * j for j in range(1, 41)] + [b"xxxxy%03d" % j for j in range(360)]
    pats += [b"xxxx", b"\xc3\xa9t\xc3"]  # 4-byte patterns: 4-byte keys; a byte >= 0x80: no byte class
    return pats + AA_WORDS + ([b"a", b"ab", b"abc", b"the"] if with_short else [])


_GQ = [b"a" * k for k in range(1, 13)] + [b" ".join([b"a"] * k) for k in range(2, 9)] + SPARSE + [b"of", b"the"]
_Q = [b"a", b"aa", b"aaa", b"a a", b"of", b"the", b"he"]  # (at most 2 matches per word: dense only as a run)
# kind -> (patterns, run unit, word unit, OLM_SHORT_LOOK, selection olm_store_inspect reports)
KINDS = {
    "GQ": (_GQ, b"a", b"a ", "0", "GQ"),
    "GQ-sx": (_GQ, b"a", b"a ", "1", "GQ"),
    "Q": (_Q, b"a", b"a ", "0", "Q"),
    "Q-sx": (_Q, b"a", b"a ", "1", "Q"),
    "C": ([b"a" * k for k in range(4, 13)] + AA_WORDS + SPARSE, b"a", b"aa ", None, "GC"),
    "G": ([b"\xe9" * k for k in range(5, 13)] + AA_WORDS + SPARSE + [b"\xc3\xa9t\xc3\xa9"], b"\xe9", b"aa ", None, "G"),
    "COOP": (_coop_patterns(False), b"x", b"aa ", None, "G+COOP"),
    "COOP-Q": (_coop_patterns(True), b"x", b"aa ", None, "GQ+COOP"),
}


def _selection(info) -> str:
    """The filter layout of scan.cu scan_launch (and launch_variant's COOP) from the staged store."""
    g, q = info["g4_bits"] > 0, info["len1"] + info["len2"] + info["len3"] > 0
    c = g and not q and info["class_run"] > 0
    return ("G" if g else "") + ("Q" if q else "") + ("C" if c else "") + ("+COOP" if info["coop"] else "")


def dense_hay(run_unit: bytes, word_unit: bytes, windowed: bool) -> bytes:
    """Sparse text with dense regions in the first chunk, in the last chunk of a tile (running into the
    next tile), in the last partial tile and -- windowed -- in the last chunk of a 4 MiB window (running
    into the next window); in both units."""
    n = (W if windowed else 0) + 40 * TILE + 1234  # tiles start at 0 and at W: the last one is partial
    hay = bytearray(tiled_text(n, 77))

    def put(at, length, unit):
        hay[at:at + length] = (unit * length)[:length]

    put(0, CHUNK, run_unit)
    put(2 * TILE, CHUNK, word_unit)
    put(5 * TILE - CHUNK, CHUNK + 88, run_unit)
    put(9 * TILE - CHUNK, CHUNK + 88, word_unit)
    put(n - 1234, CHUNK, word_unit)
    put(n - 1234 + CHUNK, 1234 - CHUNK, run_unit)
    put(20 * TILE + 100, 8, run_unit)  # a short run: a few matches
    if windowed:
        put(W - 2 * CHUNK, CHUNK, word_unit)
        put(W - CHUNK, CHUNK + 88, run_unit)
    return bytes(hay)


def dense_chunks(want: np.ndarray) -> int:
    """Source chunks that start more matches than any staging area holds."""
    if want.size == 0:
        return 0
    return int((np.bincount((want["offset"] // CHUNK).astype(np.int64)) > CHUNK_CAP_MAX).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("sf", [(0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 1)])
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_redone_chunks_on_every_scan_variant(store_cache, monkeypatch, kind, sf):
    """Every flag set, with exact statistics off and on.  OLM_SHORT_LOOK=1 gives the plain stores with
    1..3 byte patterns the second look (SX)."""
    pats, run_unit, word_unit, short_look, selection = KINDS[kind]
    path = store_cache(f"redo-{kind}", b"\n".join(pats), sf)
    info = store_info(path)
    assert _selection(info) == selection, (kind, sf, info)
    assert bool(info["flags"] & 0xE) == any(sf)
    if short_look is not None:
        monkeypatch.setenv("OLM_SHORT_LOOK", short_look)
    hay = dense_hay(run_unit, word_unit, any(sf))
    for exact in (False, True):
        o = Oracle.from_olm(path)
        with Matcher(path) as m:
            m.set_exact_stats(exact)
            for flags in DENSE_FLAGSETS:
                want = check(m, o, hay, **flags)
                if exact:
                    assert _stats(m) == _oracle_stats(o), (kind, sf, flags)
                if not flags:  # run regions: 3, and 1 at a window's end; word regions: as many
                    assert dense_chunks(want) >= (3 + any(sf)) * (1 if kind[0] == "Q" else 2) - 1, flags
                elif kind[0] != "Q" and ("word_boundary" in flags or "word_suffix" in flags):
                    assert dense_chunks(want) >= (4 if any(sf) else 3), flags


@pytest.mark.gpu
def test_redone_chunks_in_the_last_window_keep_its_extent(store_cache):
    """A normalising store without word_boundary counts the extent of each window as it scans (the
    image is brought up to date from it afterwards): redone chunks in the last window must not add their
    kept bytes twice.  The short word_boundary calls read the image around that extent."""
    sf = (0, 1, 1)
    pats = SHORT_PATS + b"\n".join(b"a" * k for k in range(1, 9))
    path = store_cache("redo-extent", pats, sf)
    win1 = bytearray(tiled_text(300_000, 6))
    for at in (0, TILE - 300, 100_000, 300_000 - 2 * CHUNK):
        win1[at:at + 2 * CHUNK] = b"a" * (2 * CHUNK)
    hay = tiled_text(W, 5) + bytes(win1)
    extent = len(Oracle.transform(bytes(win1), *sf)[0])
    shorts = [b"q" * (extent + d - 3) + b" ab" for d in (-2, 0, 1, 2, 5, 40)]
    dependent = _image_dependent(sf, hay, {}, shorts)
    assert dependent, "no short call depends on the image"
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        assert dense_chunks(check(m, o, hay)) >= 4
        for short in dependent:
            check(m, o, short, word_boundary=True)


@pytest.mark.gpu
def test_records_whose_length_needs_23_bits(store_cache):
    """A record of 2^23 + 5 source bytes does not fit a staged entry (pos << 23 | len): its chunk is
    redone.  One of 2^23 - 1 bytes does fit.  Each is planted twice, once across a tile edge."""
    rng = np.random.default_rng(23)
    letters = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz", dtype=np.uint8)
    big = rng.choice(letters, size=(1 << 23) + 5).tobytes()
    fit = rng.choice(letters, size=(1 << 23) - 1).tobytes()
    path = store_cache("redo-23bits", b"\n".join([big, fit, b"the", b"shall"]))
    up = lambda x: (x + TILE - 1) // TILE * TILE  # noqa: E731
    at_big = [1000, up(1000 + len(big) + 100) - 7]
    at_fit = [at_big[1] + len(big) + 1000]
    at_fit.append(up(at_fit[0] + len(fit) + 100) - 5)
    hay = bytearray(tiled_text(at_fit[1] + len(fit) + 3000, 9))
    for a in at_big:
        hay[a:a + len(big)] = big
    for a in at_fit:
        hay[a:a + len(fit)] = fit
    hay = bytes(hay)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        want = check(m, o, hay)
        assert int((want["len"] == len(big)).sum()) == 2 and int((want["len"] == len(fit)).sum()) == 2
        check(m, o, hay, longest_only=True, no_overlap=True)
        check(m, o, hay, word_boundary=True)
