"""The passes that run on records after the scan, driven directly with synthetic records at the sizes
where their multi-block algorithms change shape -- needs a B200.

Each pass is a multi-block algorithm with internal boundaries that scan output from a few MiB of text
never reaches: the sort's 2 048 records per warp and its histogram scan whose one-block top phase loops
past 8 388 608 records, no_overlap's 2 048 records per block and its top scan past 524 288, the
listing's 256 records per block and its top scan past 262 144, the counting table's 2 048 slots, the
newline scan's 128 MiB aggregate blocks, the 64 KiB line tiles and the matching-lines scan past 524 288
positions.  Every case compares the whole output with a plain numpy (or torch) reference.

Records are n x 3 int64 tensors: offset, len | pad << 32, ptr (the 24-byte record of
include/olm_b200.h).  Offsets of 2^63 or more are stored as their two's-complement int64; the
references work in numpy uint64.
"""
import time

import numpy as np
import pytest

import inputs
from omega_match_b200 import Matcher
from test_gpu_lines import _device_u64, _rle
from test_gpu_parity import _DevBytes
from test_lines_cpu import positions

pytestmark = pytest.mark.gpu

MIB = 1 << 20
TILE = 64 * 1024  # lines.cuh kLineTileBytes
U32 = np.uint64(0xFFFFFFFF)


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def small_store(store_cache):
    return store_cache("record-passes", b"abcde\nab\nq\n")


def _records(off, ln, pad, ptr) -> np.ndarray:
    """n x 3 uint64 records: offset, len | pad << 32, ptr"""
    rec = np.zeros((len(off), 3), dtype=np.uint64)
    rec[:, 0] = off
    rec[:, 1] = np.asarray(ln, dtype=np.uint64) | (np.asarray(pad, dtype=np.uint64) << np.uint64(32))
    rec[:, 2] = ptr
    return rec


def _to_dev(torch, rec: np.ndarray):
    return torch.from_numpy(np.ascontiguousarray(rec).view(np.int64)).cuda()


def _to_host(t) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def _first_diff(got: np.ndarray, want: np.ndarray) -> str:
    if got.shape != want.shape:
        return f"shape {got.shape} != {want.shape}"
    bad = np.flatnonzero((got != want).reshape(got.shape[0], -1).any(axis=1))
    return f"{bad.size} rows differ, first at {bad[:3]}: {got[bad[:2]].tolist()} vs {want[bad[:2]].tolist()}"


# ---- sort (radix_sort.cu) -------------------------------------------------------------------------

def _sort_keys(kind: str, n: int, rng):
    """(offsets uint64, lengths uint32) of one key distribution"""
    if kind == "random":  # every byte of offset and ~len varies: all twelve passes
        return rng.integers(0, 1 << 64, n, dtype=np.uint64), rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    if kind == "ties":  # few distinct keys: stability decides the order
        off = (rng.integers(0, 6, n, dtype=np.uint64) << np.uint64(40)) | rng.integers(0, 3, n, dtype=np.uint64)
        return off, rng.choice(np.array([3, 5, 0x10005], dtype=np.uint32), n)
    if kind == "all_equal":  # every pass skipped
        return np.full(n, 0xDEADBEEF12345678, dtype=np.uint64), np.full(n, 7, dtype=np.uint32)
    if kind == "one_byte":  # one pass (odd): the result is copied back from the scratch buffer
        return np.uint64(0x0123456789000000) | (rng.integers(0, 256, n, dtype=np.uint64) << np.uint64(24)), \
            np.full(n, 9, dtype=np.uint32)
    if kind == "two_bytes":  # one ~len pass and one offset pass (even)
        off = np.uint64(0x7700000000000042) | (rng.integers(0, 256, n, dtype=np.uint64) << np.uint64(48))
        return off, (np.uint32(5) | (rng.integers(0, 256, n, dtype=np.uint32) << np.uint32(16))).astype(np.uint32)
    off, ln = _sort_keys("random", n, rng)
    off[: n // 3] = off[n // 3: 2 * (n // 3)]  # (some equal offsets with different lengths)
    order = np.lexsort((~ln, off))
    if kind == "reverse":
        order = order[::-1]
    return off[order], ln[order]


SORT_SIZES = [0, 1, 2, 31, 32, 33, 2047, 2048, 2049, 16383, 16384, 16385, 32769]
SORT_BIG = [8_388_607, 8_388_608, 8_388_609, 9_000_001]  # the histogram scan's top block loops from 8 388 609
SORT_KINDS = ["random", "ties", "all_equal", "one_byte", "two_bytes", "sorted", "reverse"]


@pytest.mark.parametrize("kind,n", [(k, n) for k in SORT_KINDS for n in SORT_SIZES] +
                         [(k, n) for k in ("random", "ties", "one_byte") for n in SORT_BIG])
def test_sort(torch, small_store, kind, n):
    """olm_cuda_sort_records = a stable sort by (offset ascending, len descending), matcher.c:258-325:
    ties keep their input order and all 24 bytes travel with their key."""
    rng = np.random.default_rng(n * 31 + SORT_KINDS.index(kind))
    off, ln = _sort_keys(kind, n, rng)
    rec = _records(off, ln, np.arange(n, dtype=np.uint64), rng.integers(0, 1 << 64, n, dtype=np.uint64))
    want = rec[np.lexsort((~ln, off))]
    dev = _to_dev(torch, rec)
    with Matcher(small_store) as m:
        m.sort_records_device(dev.data_ptr(), n)
    got = _to_host(dev)
    assert (got == want).all(), f"{kind} n={n}: " + _first_diff(got, want)


# ---- no_overlap (filters.cu) ----------------------------------------------------------------------

def _overlap_shape(shape: str, n: int, rng):
    """sorted (offset ascending, len descending) offsets and lengths"""
    if shape == "chain":  # offset k, len 2: no certain start after record 0, one chain through every block
        return np.arange(n, dtype=np.uint64), np.full(n, 2, dtype=np.uint64)
    if shape == "long_first":  # one record over half the array, then dense short ones
        off = np.arange(n, dtype=np.uint64)
        ln = rng.integers(1, 4, n, dtype=np.uint64)
        ln[:1] = max(n // 2, 1)
        return off, ln
    if shape == "disjoint":
        ln = rng.integers(1, 9, n, dtype=np.uint64)
        gap = rng.integers(0, 3, n, dtype=np.uint64)
        return np.cumsum(ln + gap) - ln, ln
    # several lengths at each offset, distinct and descending
    group = rng.integers(1, 6, n)
    starts = np.repeat(np.cumsum(rng.integers(1, 5, group.size, dtype=np.uint64)), group)[:n]
    rank = (np.arange(group.sum()) - np.repeat(np.cumsum(group) - group, group))[:n]
    size = np.repeat(group, group)[:n]
    ln = (size - rank).astype(np.uint64) * np.uint64(2) + np.repeat(rng.integers(0, 2, group.size), group)[:n].astype(np.uint64)
    base = {"many_lengths": 0, "above_2_32": (1 << 32) - 1000, "near_2_63": (1 << 63) - 3 * n}[shape]
    return starts + np.uint64(base), ln


def _check_no_overlap(rec: np.ndarray, got: np.ndarray, what: str):
    """The greedy rule of olm_oracle.c filter_no_overlap, vectorised: record i is kept exactly when its
    offset is at or past the end of the last kept record before it (the kept set read from the pads)."""
    n = rec.shape[0]
    kept = (got[:, 1] >> np.uint64(32)).astype(np.int64)
    assert n == 0 or kept.size, f"{what}: nothing kept"
    assert (np.diff(kept) > 0).all(), f"{what}: kept records out of order"
    assert (got == rec[kept]).all(), f"{what}: kept records altered"
    off, end = rec[:, 0], rec[:, 0] + (rec[:, 1] & U32)
    prev = np.searchsorted(kept, np.arange(n), side="left") - 1
    prev_end = np.where(prev >= 0, end[kept[np.maximum(prev, 0)]], np.uint64(0))
    want = (prev < 0) | (off >= prev_end)
    keep = np.zeros(n, dtype=bool)
    keep[kept] = True
    bad = np.flatnonzero(keep != want)
    assert bad.size == 0, f"{what}: keep flag wrong at {bad[:5]} (kept {keep[bad[:5]]})"


OVERLAP_SIZES = [0, 1, 2, 2047, 2048, 2049, 524_287, 524_288, 524_289, 2_000_003]


@pytest.mark.parametrize("shape", ["chain", "long_first", "disjoint", "many_lengths", "above_2_32", "near_2_63"])
def test_no_overlap(torch, small_store, shape):
    rng = np.random.default_rng(len(shape))
    with Matcher(small_store) as m:
        for n in OVERLAP_SIZES:
            off, ln = _overlap_shape(shape, n, rng)
            rec = _records(off, ln, np.arange(n, dtype=np.uint64), rng.integers(0, 1 << 64, n, dtype=np.uint64))
            order = np.lexsort((~ln, off))
            assert (order == np.arange(n)).all(), "inputs are sorted"
            dev = _to_dev(torch, rec)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            k = m.no_overlap_device(dev.data_ptr(), n)
            ms = (time.perf_counter() - t0) * 1e3
            if shape == "chain" and n > 1_000_000:
                print(f"no_overlap single chain of {n} records ({k} kept): {ms:.1f} ms "
                      f"on {torch.cuda.get_device_name()}")
            _check_no_overlap(rec, _to_host(dev[:k]), f"{shape} n={n}")


# ---- the listing (format.cu) ----------------------------------------------------------------------

def test_listing_every_offset_width(torch, small_store):
    """"offset:bytes\\n" per record (main.c:89-133: the bytes stop at a NUL) for offsets of 1 to 20
    decimal digits, one call of over 262 144 records (the top scan loops) and sizes that are not
    multiples of the 256-record block.  The records lie inside one device buffer; each call has its own
    offset0, the offset of the buffer's first byte."""
    rng = np.random.default_rng(20)
    size = MIB + 13
    buf = rng.integers(1, 256, size, dtype=np.uint8)
    nul = np.sort(rng.choice(size, size // 150, replace=False))
    buf[nul] = 0
    hb = buf.tobytes()
    dev = torch.zeros(size + 64, dtype=torch.uint8, device="cuda")
    dev[:size] = torch.from_numpy(buf).cuda()
    calls = [(0, 1_000_003), (0, 0), (0, 1), (7, 2)] + [(10 ** k - 777, 5003) for k in range(4, 20)] + \
        [((1 << 32) - 333, 4099), ((1 << 64) - size - 1, 2305)]
    widths = set()
    with Matcher(small_store) as m:
        for offset0, n in calls:
            ln = rng.integers(1, 301, n)
            p = rng.integers(0, size - ln + 1)
            at_nul = nul[nul < size - 300][: n // 10]
            p[: at_nul.size] = at_nul  # a NUL at byte 0
            if n > 100:  # every width of the call: 1 to 4 digits from offset0 0, both sides of 10^k otherwise
                p[-8:] = [0, 5, 10, 99, 776, 777, 999, 1000]
            offs = np.uint64(offset0) + p.astype(np.uint64)
            rec = _records(offs, ln, rng.integers(0, 1 << 32, n, dtype=np.uint64), rng.integers(0, 1 << 64, n, dtype=np.uint64))
            recd = _to_dev(torch, rec)
            tptr, tlen = m.format_records_device(recd.data_ptr(), n, dev.data_ptr(), offset0)
            got = bytes(torch.as_tensor(_DevBytes(tptr, tlen), device="cuda").cpu().numpy()) if tlen else b""
            want = b"".join(b"%d:%s\n" % (o, hb[q:q + k].split(b"\0")[0])
                            for o, q, k in zip(offs.tolist(), p.tolist(), ln.tolist()))
            if got != want:
                i = next(i for i in range(min(len(got), len(want))) if got[i] != want[i])
                pytest.fail(f"offset0 {offset0} n={n}: text differs at byte {i}: {got[i - 40:i + 40]!r} vs "
                            f"{want[i - 40:i + 40]!r}")
            widths |= {len(str(o)) for o in offs.tolist()}
    assert widths == set(range(1, 21))


# ---- counts from pads (pattern_ids.cu, count_records) ---------------------------------------------

@pytest.mark.parametrize("table", [None, "0", "1"])
def test_count_records_from_pads(torch, store_cache, monkeypatch, table):
    """counts[id] += records whose pad is id, against torch.bincount, with either histogram:
    one id, ids spread over all 100 000 patterns (about 8 000 per block: the 2 048-slot block table
    fills and adds fall back to global adds), exactly 2 048 and 2 049 hot ids, and a skew."""
    if table is None:
        monkeypatch.delenv("OLM_COUNT_TABLE", raising=False)
    else:
        monkeypatch.setenv("OLM_COUNT_TABLE", table)  # read when the matcher is created
    path = store_cache("cfg5-100k", b"\n".join(inputs.synth_long_patterns(100_000)))
    g = torch.Generator(device="cuda").manual_seed(5)
    big = 20_000_003
    with Matcher(path) as m:
        P = m.pattern_count
        assert P == 100_000
        perm = torch.randperm(P, generator=g, device="cuda")
        hot = lambda k: perm[:k][torch.randint(0, k, (big,), generator=g, device="cuda")]  # noqa: E731
        cases = {
            "none": torch.zeros(0, dtype=torch.int64, device="cuda"),
            "one": torch.tensor([P - 1], device="cuda"),
            "two": torch.tensor([0, P - 1], device="cuda"),
            "single id 0": torch.zeros(100_003, dtype=torch.int64, device="cuda"),
            "single id P-1": torch.full((big,), P - 1, dtype=torch.int64, device="cuda"),
            "single id 0, many": torch.zeros(big, dtype=torch.int64, device="cuda"),
            "uniform": torch.randint(0, P, (big,), generator=g, device="cuda"),
            "2048 hot": hot(2048),
            "2049 hot": hot(2049),
            "skew": perm[(P * torch.rand(big, generator=g, device="cuda") ** 4).long().clamp_(max=P - 1)],
        }
        for name, ids in cases.items():
            n = ids.numel()
            rec = torch.zeros((n, 3), dtype=torch.int64, device="cuda")
            rec[:, 0] = torch.arange(n, device="cuda") * 3
            rec[:, 1] = 7 | (ids << 32)
            counts = torch.randint(0, 1000, (P,), generator=g, device="cuda")
            want = counts + torch.bincount(ids, minlength=P)
            m.count_records_device(rec.data_ptr(), n, counts.data_ptr())
            bad = torch.nonzero(counts != want).flatten()
            assert bad.numel() == 0, f"{name}: {bad.numel()} counts differ, first ids {bad[:5].tolist()}"
        rec = torch.zeros((1000, 3), dtype=torch.int64, device="cuda")
        rec[:, 1] = 7 | (torch.arange(1000, device="cuda") << 32)
        counts = torch.zeros(P, dtype=torch.int64, device="cuda")
        for bad_id in (P, 0xFFFFFFFF):
            v = 7 | (bad_id << 32)
            rec[999, 1] = v - (1 << 64) if v >= 1 << 63 else v
            with pytest.raises(RuntimeError):
                m.count_records_device(rec.data_ptr(), 1000, counts.data_ptr())


# ---- newline facts (lines.cu) ---------------------------------------------------------------------

def _placements(L: int):
    last_tile = (L - 1) // TILE * TILE
    edge = 128 * MIB  # 2 048 tiles: the first tile of the second aggregate block
    places = {
        "none": [],
        "first tile": [0, 5, TILE - 1],
        "last tile": sorted({last_tile, (last_tile + L - 1) // 2}),
        "last byte": [L - 1],
        "around 128 MiB": [p for p in (edge - TILE, edge - 1, edge, edge + 1) if p < L],
        "random": np.unique(np.random.default_rng(L).integers(0, L, 1000)),
        "dense": np.arange(0, L, 7),
    }
    return {k: np.asarray(v, dtype=np.int64) for k, v in places.items()}


@pytest.mark.parametrize("L", [128 * MIB - 1, 128 * MIB, 128 * MIB + 1, 128 * MIB + TILE + 1])
def test_newline_facts_across_the_aggregate_block_edge(torch, small_store, L):
    """The facts of the bytes [0, L) around 128 MiB, where the tile scan's second aggregate block
    starts, and the line of records on both sides of it.  A '\\n' just past L is not counted."""
    edge = 128 * MIB
    size = 128 * MIB + 2 * TILE
    dev = torch.full((size,), ord("a"), dtype=torch.uint8, device="cuda")
    recs = np.unique(np.array([0, TILE - 1, TILE, edge - TILE - 1, edge - 1, edge, edge + 1, L - 2, L - 1]))
    recs = recs[recs < L].astype(np.uint64)
    rec = _to_dev(torch, _records(recs, np.ones(recs.size), 0, 0))
    pos = torch.zeros((recs.size, 3), dtype=torch.int64, device="cuda")
    with Matcher(small_store) as m:
        for name, nl in _placements(L).items():
            dev[:] = ord("a")
            dev[torch.from_numpy(nl).cuda()] = 10
            dev[L] = 10
            torch.cuda.synchronize()
            want = (nl.size, int(nl[0]), int(nl[-1])) if nl.size else (0, None, None)
            assert m.newline_facts_device(dev.data_ptr(), L) == want, f"L={L} {name}"
            m.line_positions_device(rec.data_ptr(), recs.size, dev.data_ptr(), 0, L, pos.data_ptr())
            hay = np.full(L, ord("a"), dtype=np.uint8)
            hay[nl] = 10
            ref = positions(hay, recs)
            got = _to_host(pos)
            assert (got == ref).all(), f"L={L} {name}: " + _first_diff(got, ref)


def test_newline_facts_past_32_gib(torch, small_store):
    """More than 256 aggregate blocks of 128 MiB: the top scan's forward and backward loops take a
    second step.  '\\n' only in the first and the last aggregate block; a record in between gets its
    line end from the last block, carried backward over more than 256 aggregates."""
    if torch.cuda.mem_get_info()[0] < 40 << 30:
        pytest.skip("needs 40 GiB of free device memory")
    L = (32 << 30) + 128 * MIB + 12345
    dev = torch.zeros(L + 64, dtype=torch.uint8, device="cuda")
    nl = [100, 5 * MIB, L - 1000, L - 1]
    dev[torch.tensor(nl, device="cuda")] = 10
    offs = np.array([0, 100, 64 * MIB, 16 << 30, (32 << 30) + 1, L - 2000, L - 1000, L - 999, L - 1], dtype=np.uint64)
    rec = _to_dev(torch, _records(offs, np.ones(offs.size), 0, 0))
    pos = torch.zeros((offs.size, 3), dtype=torch.int64, device="cuda")
    with Matcher(small_store) as m:
        assert m.newline_facts_device(dev.data_ptr(), L) == (4, 100, L - 1)
        m.line_positions_device(rec.data_ptr(), offs.size, dev.data_ptr(), 0, L, pos.data_ptr())
    nla = np.array(nl, dtype=np.int64)
    i = np.searchsorted(nla, offs.astype(np.int64))
    pad = np.concatenate([[-1], nla, [L]])
    want = np.stack([i, pad[i] + 1, pad[i + 1]], axis=1).astype(np.uint64)
    got = _to_host(pos)
    assert (got == want).all(), _first_diff(got, want)
    del dev
    torch.cuda.empty_cache()


# ---- line positions with an origin (lines.cu) -----------------------------------------------------

def _line_bytes(kind: str, rng):
    """5 tiles and 777 bytes: a few '\\n' in tile 0, none in tiles 1 and 3, dense in tile 2, two at the
    edges of tile 4, one before the last byte; or no '\\n' at all"""
    size = 5 * TILE + 777
    hay = np.full(size, ord("a"), dtype=np.uint8)
    if kind == "mixed":
        hay[[300, 301, 40000]] = 10
        hay[2 * TILE: 3 * TILE: 3] = 10
        hay[2 * TILE + rng.integers(0, TILE, 2000)] = 10
        hay[[4 * TILE, 5 * TILE - 1, size - 2]] = 10
    return hay


@pytest.mark.parametrize("bytes_begin", [(1 << 32) + 12345, 1 << 40])
@pytest.mark.parametrize("kind", ["mixed", "no_newline"])
def test_line_positions_with_an_origin_beyond_2_32(torch, small_store, bytes_begin, kind):
    """Records of one range of a larger haystack: line, begin and end in global coordinates, past 2^32.
    Every byte of one tile (65 536 records in one block), '\\n' bytes themselves, tiles without '\\n',
    the last byte."""
    rng = np.random.default_rng(bytes_begin % 1000)
    hay = _line_bytes(kind, rng)
    size = hay.size
    local = np.concatenate([np.arange(2 * TILE, 3 * TILE), rng.integers(TILE, 2 * TILE, 300),
                            rng.integers(3 * TILE, 4 * TILE, 300), np.flatnonzero(hay == 10),
                            [0, 1, TILE - 1, TILE, 4 * TILE - 1, 4 * TILE, 4 * TILE + 1, size - 2, size - 1]])
    local = np.sort(local).astype(np.uint64)
    origin = ((1 << 33) + 5, bytes_begin - 4321, bytes_begin + size + 99)
    dev = torch.zeros(size + 64, dtype=torch.uint8, device="cuda")
    dev[:size] = torch.from_numpy(hay).cuda()
    rec = _to_dev(torch, _records(local + np.uint64(bytes_begin), np.full(local.size, 4), 0, 0))
    pos = torch.zeros((local.size, 3), dtype=torch.int64, device="cuda")
    with Matcher(small_store) as m:
        m.line_positions_device(rec.data_ptr(), local.size, dev.data_ptr(), bytes_begin, size, pos.data_ptr(),
                                origin=origin)
    # the origin arithmetic of test_lines_cpu.test_line_origins_against_the_reference
    ref = positions(hay, local)
    i, c, b = ref[:, 0], np.uint64((hay == 10).sum()), np.uint64(bytes_begin)
    want = np.stack([np.uint64(origin[0]) + i, np.where(i > 0, b + ref[:, 1], np.uint64(origin[1])),
                     np.where(i < c, b + ref[:, 2], np.uint64(origin[2]))], axis=1)
    got = _to_host(pos)
    assert (got == want).all(), _first_diff(got, want)


# ---- matching lines (lines.cu) --------------------------------------------------------------------

def _line_runs(shape: str, n: int, rng):
    """non-decreasing positions (n x 3: line, begin, end) of one shape"""
    if shape == "one_line":
        line = np.zeros(n, dtype=np.uint64)
    elif shape in ("own_lines", "beyond_2_32"):
        line = np.cumsum(rng.integers(1, 3, n, dtype=np.uint64)) - np.uint64(1)
    else:  # runs that start and end exactly at the 2 048-position block edges, and one over several blocks
        head = rng.random(n) < 0.01
        for e in range(2048, n, 2048):
            head[e - 2: e + 3] = False
            k = e // 2048 % 4  # a run starts at the edge, straddles it, is one record before it, starts after it
            head[[e] if k == 0 else [] if k == 1 else [e - 1, e] if k == 2 else [min(e + 1, n - 1)]] = True
        head[5000:12000] = False  # one run over several blocks
        head[:1] = True
        line = (np.cumsum(head) - 1).astype(np.uint64)
    base = np.uint64((1 << 32) - 3 if shape == "beyond_2_32" else 17)
    line = line + base
    return np.stack([line, line * np.uint64(10), line * np.uint64(10) + np.uint64(9)], axis=1)


@pytest.mark.parametrize("shape", ["one_line", "own_lines", "block_edges", "beyond_2_32"])
def test_matching_lines_device(torch, small_store, shape):
    rng = np.random.default_rng(len(shape) + 3)
    with Matcher(small_store) as m:
        for n in [0, 1, 2, 2047, 2048, 2049, 4097, 524_287, 524_288, 524_289, 2_000_003]:
            pos = _line_runs(shape, n, rng)
            dev = _to_dev(torch, pos)
            n_lines, lp = m.matching_lines_device(dev.data_ptr(), n)
            got, want = _device_u64(torch, lp, n_lines, 4), _rle(pos)
            assert got.shape == want.shape and (got == want).all(), f"{shape} n={n}: " + _first_diff(got, want)
