"""Lines (include/olm_b200.h "lines"): the line of every record and the matching lines of a call,
computed on the GPU -- needs a B200.

The expected records come from the CPU oracle, the expected positions from the numpy reference of
test_lines_cpu (searchsorted over the haystack's '\\n' bytes).
"""
import ctypes as C
import time

import numpy as np
import pytest

import inputs
from omega_match_b200 import Matcher
from omega_match_b200.omega_match import LINE_POS_DTYPE, _flag_ints
from omega_match_b200.sharding import line_origins, shard_plan
from oracle.oracle import Oracle
from test_gpu_multi import _devices
from test_gpu_pattern_ids import EDGE_FLAGSETS
from test_lines_cpu import positions

pytestmark = pytest.mark.gpu

MIB = 1 << 20
TILE = 64 * 1024  # lines.cuh kLineTileBytes
PATTERNS = [b"a", b"ab", b"abcde", b"hello world", b"line", b"end", b"q", b"x y"]


def _rle(pos: np.ndarray) -> np.ndarray:
    """matching lines of positions (n x 3: line, begin, end) -> m x 4 (line, begin, end, records)"""
    if pos.shape[0] == 0:
        return np.zeros((0, 4), dtype=np.uint64)
    head = np.flatnonzero(np.concatenate([[True], pos[1:, 0] != pos[:-1, 0]]))
    out = np.zeros((head.size, 4), dtype=np.uint64)
    out[:, :3] = pos[head]
    out[:, 3] = np.diff(np.concatenate([head, [pos.shape[0]]]))
    return out


def _as3(a) -> np.ndarray:
    return np.stack([a["line"], a["line_begin"], a["line_end"]], axis=1).astype(np.uint64) if "line_begin" in a.dtype.names \
        else np.stack([a["line"], a["begin"], a["end"]], axis=1).astype(np.uint64)


def _as4(lines) -> np.ndarray:
    return np.stack([lines["line"], lines["begin"], lines["end"], lines["records"]], axis=1).astype(np.uint64)


def _check(m: Matcher, hay: bytes, want=None, what="", **flags):
    """match_lines / matching_lines against `want` (the oracle's records, or match_arrays) + the reference."""
    arr = np.frombuffer(hay, dtype=np.uint8)
    if want is None:
        want = m.match_arrays(hay, **flags)
    got = m.match_lines(hay, **flags)
    assert got.size == want.size and (got["offset"] == want["offset"]).all() and (got["len"] == want["len"]).all(), \
        f"{what} {flags}: records differ ({got.size} vs {want.size})"
    ref = positions(arr, got["offset"])
    bad = np.flatnonzero((_as3(got) != ref).any(axis=1))
    assert bad.size == 0, f"{what} {flags}: positions differ at {bad[:5]}: {_as3(got)[bad[:3]]} vs {ref[bad[:3]]}"
    lines = m.matching_lines(hay, **flags)
    assert (_as4(lines) == _rle(ref)).all() and lines.size == _rle(ref).shape[0], f"{what} {flags}: matching lines"
    assert int(lines["records"].sum()) == got.size
    return got


# ---- against the oracle, every store-flag set ---------------------------------------------------

def _edge_haystacks():
    hays = [b"", b"abcde", b"\n", b"\n" * 40, b"ab\r\nab\r\n\r\nab", b"ab\rab\r\rab", b"abcde\nab\nab", b"\nab\n\nabcde",
            b"hello\nworld\nhello  \n world x\ny", b"end\nend\nline end", b"q" * 5 + b"\n" + b"q" * 300 + b"\nq"]
    for t in (TILE, 2 * TILE):  # '\n' around tile edges
        for d in (-16, -1, 0, 1, 16):
            h = bytearray(b"ab cd " * ((t + 64) // 6))
            h[t + d] = 10
            h[t - 20] = 10
            hays.append(bytes(h))
    h = bytearray(b"abcde line " * (3 * TILE // 11))
    for p in range(TILE - 40, TILE + 40, 3):
        h[p] = 10
    hays.append(bytes(h))
    return hays


@pytest.mark.parametrize("sf", inputs.STORE_FLAG_SETS)
def test_lines_on_edge_haystacks(store_cache, sf):
    buf = b"\n".join(p for p in PATTERNS if inputs.py_normalize(p, *sf))
    path = store_cache("lines-edge", buf, sf)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        for hay in _edge_haystacks():
            for flags in EDGE_FLAGSETS:
                _check(m, hay, o.match(hay, **flags), f"{sf} n={len(hay)}", **flags)
                counts = m.pattern_counts(hay, **flags)
                assert int(counts.sum()) == int(m.matching_lines(hay, **flags)["records"].sum())


def test_elide_whitespace_match_across_a_newline_reports_its_first_line(store_cache):
    path = store_cache("lines-ew", b"hello world\n", (0, 0, 1))
    hay = b"say hello\n  world\nhello world"
    with Matcher(path) as m:
        got = _check(m, hay, Oracle.from_olm(path).match(hay))
        assert got["offset"].tolist() == [4, 18] and got["line"].tolist() == [0, 2]
        assert got["line_end"][0] == 9


def test_records_equal_match_arrays_with_ids_on_and_off(store_cache):
    names = inputs.case_patterns(dict(patterns="names", store_flags=(1, 1, 1)))
    path = store_cache("lines-names-111", names, (1, 1, 1))
    hay = inputs.text_haystack(3 * MIB + 7, 11).tobytes()
    with Matcher(path) as m:
        for flags in ({}, {"longest_only": True, "no_overlap": True, "word_boundary": True}):
            off = _check(m, hay, **flags)
            assert "pattern_id" not in off.dtype.names
            ids = m.match_ids(hay, **flags)
            m.set_pattern_ids(True)
            on = _check(m, hay, **flags)
            m.set_pattern_ids(False)
            assert (on["pattern_id"] == ids["pattern_id"]).all()
            assert (_as3(on) == _as3(off)).all()


# ---- long lines and dense newlines ---------------------------------------------------------------

def test_64_mib_single_line_and_a_newline_every_byte(store_cache):
    path = store_cache("lines-long", b"abcde\nab\nq\n")
    n = 64 * MIB
    one = np.frombuffer(b"xabcdexqx" * (n // 9 + 1), dtype=np.uint8)[:n].copy()
    with Matcher(path) as m:
        t0 = time.perf_counter()
        got = _check(m, one.tobytes(), what="single line")
        wall = time.perf_counter() - t0
        t = m.last_timing()
        assert got.size > 10_000_000 and (got["line"] == 0).all() and (got["line_end"] == n).all()
        print(f"single line of {n} bytes, {got.size} records: total_ms {t['total_ms']:.3f}, scan_ms {t['scan_ms']:.3f}, "
              f"wall (both calls) {wall:.2f} s")
        dense = one.copy()
        dense[1::2] = 10  # '\n' every other byte: 'a' 'q' records all start right after one
        _check(m, dense.tobytes(), what="dense")
        every = np.full(n, 10, dtype=np.uint8)
        every[::7] = ord("q")
        got = _check(m, every.tobytes(), what="every byte")
        assert got.size == n // 7 + (n % 7 > 0)


# ---- spans, shards, several GPUs ---------------------------------------------------------------

def _span_haystack(n: int, seed: int) -> bytes:
    hay = inputs.text_haystack(n, seed)
    hay[hay == 10] = 32
    rng = np.random.default_rng(seed)
    for p in rng.integers(0, n, 300):  # short lines, some crossing span edges ...
        hay[p] = 10
    hay[4 * MIB - 1] = 10
    hay[4 * MIB + 100:12 * MIB] = np.where(hay[4 * MIB + 100:12 * MIB] == 10, 32, hay[4 * MIB + 100:12 * MIB])
    for edge in range(4 * MIB, n - 6, 4 * MIB):  # ... one line longer than a span, matches on span edges
        hay[edge - 5:edge + 6] = np.frombuffer(b"Christopher", dtype=np.uint8)
    return hay.tobytes()


def test_host_span_path(store_cache, monkeypatch):
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    hay = _span_haystack(17 * MIB + 12345, 5)
    for sf in ((0, 0, 0), (1, 1, 1)):
        path = store_cache("span-names", names, sf)
        with Matcher(path) as whole:
            wants = {i: whole.match_arrays(hay, **kw) for i, kw in enumerate(({}, {"no_overlap": True},
                                                                               {"longest_only": True, "no_overlap": True}))}
        monkeypatch.setenv("OLM_HOST_SPAN_BYTES", str(4 * MIB))
        with Matcher(path) as m:
            for i, kw in enumerate(({}, {"no_overlap": True}, {"longest_only": True, "no_overlap": True})):
                _check(m, hay, wants[i], f"span {sf}", **kw)
            _check(m, b"no newline here abc " * 300_000, what="span, one line")
        monkeypatch.delenv("OLM_HOST_SPAN_BYTES")


@pytest.mark.parametrize("sf", [(0, 0, 0), (1, 1, 1)])
def test_multi_matcher_lines(store_cache, sf):
    names = inputs.case_patterns(dict(patterns="names", store_flags=sf))
    path = store_cache("multi-names", names, sf)
    hay = _span_haystack(13 * MIB + 4321, 31)
    with Matcher(path) as one, Matcher(path, devices=_devices(2)) as many:
        for kw in ({}, {"no_overlap": True}, {"longest_only": True, "no_overlap": True}):
            _check(many, hay, one.match_arrays(hay, **kw), f"multi {sf}", **kw)


def test_multi_matcher_lines_with_window_tails(store_cache):
    sf = (1, 1, 1)
    path = store_cache("counts-tails", b"\n".join([b"ab", b"the", b"king", b"lord", b"of", b"and", b"jesus"]), sf)
    hay = inputs.text_haystack(9 * 4 * MIB + 77, 3).tobytes()
    with Matcher(path) as one, Matcher(path, devices=_devices(2)) as many:
        for kw in ({"word_boundary": True}, {"word_boundary": True, "longest_only": True, "no_overlap": True}):
            _check(many, hay, one.match_arrays(hay, **kw), "tails", **kw)


@pytest.mark.parametrize("kind", ["plain", "windowed"])
def test_shards_one_after_another_on_one_gpu(store_cache, kind):
    """olm_cuda_match_shard + newline facts of the own range + line_origins + line positions per shard:
    the concatenation equals the whole haystack's positions."""
    torch = pytest.importorskip("torch")
    from test_gpu_parity import _device_records
    if kind == "plain":
        pats = inputs.synth_long_patterns(3000) + [b"ab", b"the", b"o"]
        hay = inputs.plant(inputs.synth_haystack(3_000_000, 123), pats, 9, block=2048)
        hay[::977] = 10
        hay[1_000_000:2_200_000][hay[1_000_000:2_200_000] == 10] = 32  # a line across shards
        sf, largest = (0, 0, 0), 24
    else:
        pats = [p for p in inputs.golden_data("names.txt").split(b"\n") if p][::5]
        hay = inputs.text_haystack(9 * 4 * MIB + 4321, 21)
        sf, largest = (1, 1, 1), max(len(p) for p in pats)
    path = store_cache(f"lines-shard-{kind}", b"\n".join(pats), sf)
    dev = torch.zeros(hay.size + 64, dtype=torch.uint8, device="cuda")
    dev[:hay.size] = torch.from_numpy(hay).cuda()
    torch.cuda.synchronize()
    with Matcher(path) as m:
        want = positions(hay, m.match_arrays(hay)["offset"])
        for world in (1, 3, 4):
            plan = shard_plan(hay.size, world, largest, windowed=any(sf))
            recs, facts, slices = [], [], []
            for s in plan:
                ln = s.slice_end - s.slice_begin
                sl = torch.zeros(((ln + 15) // 16) * 16 + 16, dtype=torch.uint8, device="cuda")
                sl[:ln] = dev[s.slice_begin:s.slice_end]
                torch.cuda.synchronize()
                c, p = m.match_shard(sl.data_ptr(), s.slice_begin, ln, s.own_begin, s.own_end, hay.size, 0)
                recs.append(_device_records(torch, p, c).clone())
                own = sl.data_ptr() + (s.own_begin - s.slice_begin)
                facts.append(m.newline_facts_device(own, s.own_end - s.own_begin))
                slices.append((sl, own))
            origins = line_origins(facts, [(s.own_begin, s.own_end) for s in plan], hay.size)
            got = []
            for s, r, (sl, own), o in zip(plan, recs, slices, origins):
                pos = torch.zeros((max(r.shape[0], 1), 3), dtype=torch.int64, device="cuda")
                m.line_positions_device(r.data_ptr(), r.shape[0], own, s.own_begin, s.own_end - s.own_begin,
                                        pos.data_ptr(), origin=o)
                got.append(pos[:r.shape[0]].cpu().numpy().astype(np.uint64))
            got = np.concatenate(got)
            assert got.shape == want.shape and (got == want).all(), f"{kind} x{world}"


def test_device_path(store_cache):
    torch = pytest.importorskip("torch")
    names = inputs.case_patterns(dict(patterns="names", store_flags=(1, 0, 0)))
    path = store_cache("counts-names-ci", names, (1, 0, 0))
    hay = inputs.text_haystack(9 * 4 * MIB + 321, 12)
    dev = torch.zeros(hay.size + 64, dtype=torch.uint8, device="cuda")
    dev[:hay.size] = torch.from_numpy(hay).cuda()
    torch.cuda.synchronize()
    with Matcher(path) as m:
        for flags in ({}, {"longest_only": True, "no_overlap": True}):
            want = m.match_arrays(hay, **flags)
            cnt, ptr = m.match_device(dev.data_ptr(), hay.size, **flags)
            assert cnt == want.size
            pos = torch.zeros((cnt, 3), dtype=torch.int64, device="cuda")
            m.line_positions_device(ptr, cnt, dev.data_ptr(), 0, hay.size, pos.data_ptr())
            ref = positions(hay, want["offset"])
            assert (pos.cpu().numpy().astype(np.uint64) == ref).all()
            n_lines, lp = m.matching_lines_device(pos.data_ptr(), cnt)
            lines = _device_u64(torch, lp, n_lines, 4)
            assert lines.shape == _rle(ref).shape and (lines == _rle(ref)).all()
            assert m.newline_facts_device(dev.data_ptr(), hay.size) == (
                int((hay == 10).sum()), int(np.flatnonzero(hay == 10)[0]), int(np.flatnonzero(hay == 10)[-1]))


def _device_u64(torch, ptr, rows, cols):
    """copy of rows x cols uint64 words of library-owned device memory"""
    class Dev:
        __cuda_array_interface__ = {"shape": (rows, cols), "typestr": "<u8", "data": (ptr, False), "version": 2}
    return torch.as_tensor(Dev(), device="cuda").clone().cpu().numpy() if rows else np.zeros((0, cols), dtype=np.uint64)


def test_one_million_patterns_device_path(store_cache):
    """256 MiB of the cfg5 haystack (one '\\n' in 64 bytes) x 1 M patterns; the reference with torch."""
    torch = pytest.importorskip("torch")
    import synth_torch
    from test_gpu_parity import _device_records
    pats = inputs.synth_long_patterns(1_000_000)
    path = store_cache("ids-cfg5-1m", b"\n".join(pats) + b"\n")
    n = 256 * MIB
    hay = torch.zeros(n + 256, dtype=torch.uint8, device="cuda")
    hay[:n] = synth_torch.synth_haystack_torch(n, inputs.SEED_H5, device="cuda")
    pb, pl = synth_torch.pack_patterns(pats, "cuda")
    synth_torch.plant_torch(hay[:n], pb, pl, inputs.SEED_H5 ^ 0x77)
    torch.cuda.synchronize()
    with Matcher(path) as m:
        cnt, ptr = m.match_device(hay.data_ptr(), n)
        rec = _device_records(torch, ptr, cnt).clone()
        pos = torch.zeros((cnt, 3), dtype=torch.int64, device="cuda")
        m.line_positions_device(rec.data_ptr(), cnt, hay.data_ptr(), 0, n, pos.data_ptr())
        nl = torch.nonzero(hay[:n] == 10).flatten()
        assert nl.numel() > n // 128
        i = torch.searchsorted(nl, rec[:, 0].contiguous())
        pad = torch.cat([torch.tensor([-1], device="cuda"), nl, torch.tensor([n], device="cuda")])
        assert bool((pos[:, 0] == i).all()) and bool((pos[:, 1] == pad[i] + 1).all()) and bool((pos[:, 2] == pad[i + 1]).all())
        n_lines, _ = m.matching_lines_device(pos.data_ptr(), cnt)
        assert n_lines == int(torch.unique_consecutive(i).numel())


# ---- errors ----------------------------------------------------------------------------------

def test_errors(store_cache):
    torch = pytest.importorskip("torch")
    path = store_cache("lines-edge", b"\n".join(p for p in PATTERNS), (0, 0, 0))
    hay = b"ab\nab abcde\n"
    dev = torch.zeros(64, dtype=torch.uint8, device="cuda")
    dev[:len(hay)] = torch.frombuffer(bytearray(hay), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    with Matcher(path) as m:
        cnt, ptr = m.match_device(dev.data_ptr(), len(hay))
        assert cnt > 2
        pos = torch.zeros((cnt, 3), dtype=torch.int64, device="cuda")
        with pytest.raises(RuntimeError):  # records before the bytes
            m.line_positions_device(ptr, cnt, dev.data_ptr() + 16, 16, 0, pos.data_ptr(), origin=(0, 0, 0))
        with pytest.raises(RuntimeError):  # records behind them
            m.line_positions_device(ptr, cnt, dev.data_ptr(), 0, 4, pos.data_ptr())
        with pytest.raises(RuntimeError):  # no origin, but the bytes do not start at 0
            m.line_positions_device(ptr, cnt, dev.data_ptr(), 16, len(hay), pos.data_ptr())
        m.line_positions_device(ptr, cnt, dev.data_ptr(), 0, len(hay), pos.data_ptr())  # still usable
        L = m._lib
        assert L.olm_cuda_line_positions(m._matcher, ptr, cnt, dev.data_ptr(), 0, len(hay), None, None) == -1
        assert L.olm_cuda_newline_facts(m._matcher, dev.data_ptr(), len(hay), None) == -1
        assert L.olm_cuda_matching_lines_device(m._matcher, pos.data_ptr(), cnt, None, None) == -1
        n_lines, total = C.c_uint64(), C.c_uint64()
        assert L.olm_cuda_matching_lines(m._matcher, hay, len(hay), *_flag_ints({}), None, C.byref(n_lines),
                                         C.byref(total)) == -1
        assert L.olm_cuda_match_lines(m._matcher, hay, len(hay), *_flag_ints({}), None, None) == -1
        assert m.match_lines(hay).size == cnt and LINE_POS_DTYPE.itemsize == 24
