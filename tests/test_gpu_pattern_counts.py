"""Pattern counts (include/olm_b200.h "pattern counts"): how often each pattern of the store occurs,
counted on the GPU without returning the records -- needs a B200.

The expected counts come from the CPU oracle: every record of `Oracle.match` is normalised the way
the store normalises, mapped to its id through the catalogue, and the ids are counted.
"""
import ctypes as C
import random

import numpy as np
import pytest

import inputs
from omega_match_b200 import Compiler, Matcher
from omega_match_b200.omega_match import _flag_ints
from omega_match_b200.sharding import WINDOW, shard_plan
from oracle.oracle import Oracle
from test_gpu_multi import _devices
from test_gpu_pattern_ids import EDGE_FLAGSETS, _bucket_records, _device_ids, _normalised_span

pytestmark = pytest.mark.gpu

MIB = 1 << 20


def _oracle_counts(m: Matcher, o: Oracle, hay: bytes, sf, **flags):
    """(counts, records) of the oracle's match stream."""
    want = o.match(hay, **flags)
    ids = {m.pattern(i): i for i in range(m.pattern_count)}
    norm = {}
    pid = []
    for off, ln in zip(want["offset"].tolist(), want["len"].tolist()):
        span = bytes(hay[off:off + ln])
        if span not in norm:
            norm[span] = ids[_normalised_span(span, sf)]
        pid.append(norm[span])
    return np.bincount(np.array(pid, dtype=np.int64), minlength=m.pattern_count).astype(np.uint64), want.size


def _count_c(m: Matcher, hay: bytes, counts: np.ndarray, **flags) -> int:
    """olm_cuda_count_patterns into `counts` (added); returns *total."""
    buf = (C.c_char * len(hay)).from_buffer_copy(hay) if len(hay) else None
    total = C.c_uint64()
    rc = m._lib.olm_cuda_count_patterns(m._matcher, C.addressof(buf) if buf is not None else None, len(hay),
                                        *_flag_ints(flags), counts.ctypes.data, C.byref(total))
    assert rc == 0, f"olm_cuda_count_patterns failed {flags}"
    return int(total.value)


def _check_counts(m: Matcher, o: Oracle, hay, sf, **flags):
    hay = bytes(hay)
    want, n = _oracle_counts(m, o, hay, sf, **flags)
    counts = np.zeros(m.pattern_count, dtype=np.uint64)
    total = _count_c(m, hay, counts, **flags)
    assert total == n, f"{sf} {flags}: total {total}, oracle {n} records"
    assert (counts == want).all(), f"{sf} {flags}: counts differ at ids {np.nonzero(counts != want)[0][:8]}"
    assert (m.pattern_counts(hay, **flags) == want).all()
    return want


def _oracle_only(m: Matcher, path: str, hay, sf, **flags) -> np.ndarray:
    return _oracle_counts(m, Oracle.from_olm(path), bytes(hay), sf, **flags)[0]


# ---- against the oracle ----------------------------------------------------------------------

EDGE_HAYS = [b"", b"a", b"abcd", b"abcde", b"xabcdefghij", b"abcdefghij" * 3, b"x" * 41, b"x" * 450,
             b"hello world", b"Hello,  World!\n", b"the King\nline\n", b"abcd" * 1000, (b"abcde " * 7000)[:32768 + 5],
             b"q" * 32766 + b"abcdefghij", b"q" * 32760 + b"x" * 220, b"A-b-C-d-E, h.e.l.l.o \t\t w-o-r-l-d"]


@pytest.mark.parametrize("sf", inputs.STORE_FLAG_SETS)
def test_counts_on_edge_haystacks(store_cache, sf):
    from test_gpu_parity import EDGE_PATTERNS
    buf = b"\n".join(p for p in EDGE_PATTERNS if inputs.py_normalize(p, *sf)) + b"\n"
    path = store_cache("edge", buf, sf)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        for hay in EDGE_HAYS:
            for flags in EDGE_FLAGSETS:
                _check_counts(m, o, hay, sf, **flags)


@pytest.mark.parametrize("seed", range(6))
def test_counts_on_random_stores_and_haystacks(store_cache, seed):
    rng = random.Random(9100 + seed)
    alph = b"abcABC xyz.,-'\n\t_09"
    pats = set()
    while len(pats) < rng.choice([5, 40, 400]):
        pats.add(bytes(rng.choice(b"abcABC xyz.-'_09") for _ in range(rng.choice([1, 2, 2, 3, 3, 4, 4, 5, 6, 9, 14, 30]))))
    sf = inputs.STORE_FLAG_SETS[seed % len(inputs.STORE_FLAG_SETS)]
    lines = sorted(p for p in pats if inputs.py_normalize(p, *sf))
    lines += lines[::3]  # duplicates
    path = store_cache(f"counts-fuzz{seed}", b"\n".join(lines), sf)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        for i in range(8):
            n = rng.choice([0, 1, 5, 300, 4000, 40000, 70001])
            hay = bytes(rng.choice(alph) for _ in range(n))
            _check_counts(m, o, hay, sf, **EDGE_FLAGSETS[i % len(EDGE_FLAGSETS)])


def test_counts_across_window_edges(store_cache):
    hay = bytearray(b"." * (WINDOW + 100))
    hay[WINDOW - 5:WINDOW + 5] = b"helloworld"
    hay[WINDOW + 20:WINDOW + 40] = b"Hel-lo, wor ld ab  x"
    for sf in ((1, 0, 0), (1, 1, 0), (1, 1, 1), (0, 1, 0), (0, 0, 1)):
        pats = [p for p in (b"HELLOWORLD", b"hello", b"hel lo", b"ab  ", b"ab", b"zq") if inputs.py_normalize(p, *sf)]
        path = store_cache("ids-window", b"\n".join(pats), sf)
        o = Oracle.from_olm(path)
        with Matcher(path) as m:
            for flags in ({}, {"word_boundary": True}, {"longest_only": True, "no_overlap": True}):
                _check_counts(m, o, hay, sf, **flags)


# ---- skewed histograms: both variants of the counting kernel ---------------------------------

def test_single_pattern_repeated_millions_of_times(store_cache):
    path = store_cache("counts-skew", b"abcde\nzzzzzz\nab\nq\n")
    reps = 3_000_000
    hay = b"abcde" * reps
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        ids = {m.pattern(i): i for i in range(m.pattern_count)}
        for flags in ({}, {"longest_only": True, "no_overlap": True}):
            counts = np.zeros(m.pattern_count, dtype=np.uint64)
            total = _count_c(m, hay, counts, **flags)
            assert counts[ids[b"abcde"]] == reps and counts[ids[b"zzzzzz"]] == 0 and counts[ids[b"q"]] == 0
            assert counts[ids[b"ab"]] == (0 if flags else reps)
            assert total == int(counts.sum())
            assert (counts == _oracle_only(m, path, hay, (0, 0, 0), **flags)).all()
        _check_counts(m, o, hay[:200_005], (0, 0, 0))


@pytest.mark.parametrize("table", ["0", "1"])
def test_dense_names_text_with_and_without_the_block_table(store_cache, monkeypatch, table):
    """The same counts whichever histogram runs (OLM_COUNT_TABLE forces one)."""
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    path = store_cache("ids-names", names, (0, 0, 0))
    hay = inputs.text_haystack(24 * MIB + 5, 17).tobytes()
    with Matcher(path) as m:
        want = _oracle_only(m, path, hay, (0, 0, 0))
        small = _check_counts(m, Oracle.from_olm(path), hay[:3 * MIB], (0, 0, 0))
    monkeypatch.setenv("OLM_COUNT_TABLE", table)
    with Matcher(path) as m:
        assert (m.pattern_counts(hay) == want).all()
        assert (m.pattern_counts(hay[:3 * MIB]) == small).all()


def test_counts_at_one_million_patterns(store_cache):
    """256 MiB of the cfg5 haystack x 1 M patterns, device path: a bincount of the ids-on records."""
    torch = pytest.importorskip("torch")
    import synth_torch
    pats = inputs.synth_long_patterns(1_000_000)
    path = store_cache("ids-cfg5-1m", b"\n".join(pats) + b"\n")
    n = 256 * MIB
    hay = torch.zeros(n + 256, dtype=torch.uint8, device="cuda")
    hay[:n] = synth_torch.synth_haystack_torch(n, inputs.SEED_H5, device="cuda")
    pb, pl = synth_torch.pack_patterns(pats, "cuda")
    synth_torch.plant_torch(hay[:n], pb, pl, inputs.SEED_H5 ^ 0x77)
    torch.cuda.synchronize()
    with Matcher(path) as m:
        m.set_pattern_ids(True)
        cnt, ptr = m.match_device(hay.data_ptr(), n)
        _, rec = _device_ids(torch, ptr, cnt)
        want = torch.bincount((rec[:, 1] >> 32) & 0xFFFFFFFF, minlength=len(pats))
        m.set_pattern_ids(False)
        counts = torch.zeros(len(pats), dtype=torch.int64, device="cuda")
        total = m.pattern_counts_device(hay.data_ptr(), n, counts.data_ptr())
        assert total == cnt and bool((counts == want).all())
        t = m.last_timing()
        assert t["total_ms"] >= t["scan_ms"]


# ---- the interface ---------------------------------------------------------------------------

def test_counts_add_up_in_c_and_are_fresh_in_python(store_cache):
    names = inputs.case_patterns(dict(patterns="names", store_flags=(1, 1, 1)))
    path = store_cache("counts-names-111", names, (1, 1, 1))
    hay = inputs.text_haystack(2 * MIB + 3, 41).tobytes()
    with Matcher(path) as m:
        for flags in ({}, {"word_boundary": True, "longest_only": True, "no_overlap": True}):
            want = _oracle_only(m, path, hay, (1, 1, 1), **flags)
            counts = np.zeros(m.pattern_count, dtype=np.uint64)
            t1 = _count_c(m, hay, counts, **flags)
            t2 = _count_c(m, hay[:MIB], counts, **flags)
            assert (counts == want + _oracle_only(m, path, hay[:MIB], (1, 1, 1), **flags)).all()
            assert t1 == int(want.sum()) and t1 + t2 == int(counts.sum())
            a, b = m.pattern_counts(hay, **flags), m.pattern_counts(hay, **flags)
            assert a.dtype == np.uint64 and a.size == m.pattern_count
            assert (a == want).all() and (b == want).all()


def test_the_ids_setting_is_left_as_it_was(store_cache):
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    path = store_cache("ids-names", names, (0, 0, 0))
    hay = inputs.text_haystack(MIB + 7, 5)
    with Matcher(path) as m:
        before = m._match_records(hay)
        m.pattern_counts(hay)  # the first count call loads the tables, ids stay off
        after = m._match_records(hay)
        assert after.tobytes() == before.tobytes() and not after["_pad"].any()
        m.set_pattern_ids(True)
        on = m._match_records(hay)
        m.pattern_counts(hay, no_overlap=True)
        again = m._match_records(hay)
        assert again.tobytes() == on.tobytes() and on["_pad"].any()


def test_device_path_accumulates(store_cache):
    torch = pytest.importorskip("torch")
    names = inputs.case_patterns(dict(patterns="names", store_flags=(1, 0, 0)))
    path = store_cache("counts-names-ci", names, (1, 0, 0))
    hay = inputs.text_haystack(9 * WINDOW + 321, 12)
    dev = torch.zeros(hay.size + 64, dtype=torch.uint8, device="cuda")
    dev[:hay.size] = torch.from_numpy(hay).cuda()
    torch.cuda.synchronize()
    with Matcher(path) as m:
        for flags in ({}, {"word_boundary": True}, {"longest_only": True, "no_overlap": True}):
            want = torch.from_numpy(_oracle_only(m, path, hay, (1, 0, 0), **flags).astype(np.int64)).cuda()
            counts = torch.zeros(m.pattern_count, dtype=torch.int64, device="cuda")
            t1 = m.pattern_counts_device(dev.data_ptr(), hay.size, counts.data_ptr(), **flags)
            t2 = m.pattern_counts_device(dev.data_ptr(), hay.size, counts.data_ptr(), **flags)
            assert t1 == t2 == int(want.sum().item())
            assert bool((counts == 2 * want).all())


@pytest.mark.parametrize("kind", ["plain", "windowed"])
def test_shards_and_gathered_records_counted(store_cache, kind):
    torch = pytest.importorskip("torch")
    if kind == "plain":
        pats = inputs.synth_long_patterns(5000) + [b"ab", b"the", b"o", b"King"]
        hay = inputs.plant(inputs.synth_haystack(3_000_000, 123), pats, 9, block=2048)
        sf, largest = (0, 0, 0), 24
    else:
        pats = [p for p in inputs.golden_data("names.txt").split(b"\n") if p][::5]
        hay = inputs.text_haystack(9 * WINDOW + 4321, 21)
        sf, largest = (1, 1, 1), max(len(p) for p in pats)
    path = store_cache(f"shard-{kind}", b"\n".join(pats), sf)
    dev = torch.zeros(hay.size + 64, dtype=torch.uint8, device="cuda")
    dev[:hay.size] = torch.from_numpy(hay).cuda()
    torch.cuda.synchronize()
    with Matcher(path) as m:
        P = m.pattern_count
        for flags in ({}, {"longest_only": True, "word_boundary": True}):
            want = torch.from_numpy(_oracle_only(m, path, hay, sf, **flags).astype(np.int64)).cuda()
            m.set_pattern_ids(True)
            for world in (2, 4):
                for host in (False, True):
                    counts = torch.zeros(P, dtype=torch.int64, device="cuda")
                    for s in shard_plan(hay.size, world, largest, windowed=any(sf)):
                        ln = s.slice_end - s.slice_begin
                        if host:
                            hslice = np.ascontiguousarray(hay[s.slice_begin:s.slice_end])
                            c, p = m.match_shard_host(hslice.ctypes.data, s.slice_begin, ln, s.own_begin, s.own_end,
                                                      hay.size, 0, **flags)
                        else:
                            sl = torch.zeros(((ln + 15) // 16) * 16 + 16, dtype=torch.uint8, device="cuda")
                            sl[:ln] = dev[s.slice_begin:s.slice_end]
                            torch.cuda.synchronize()
                            c, p = m.match_shard(sl.data_ptr(), s.slice_begin, ln, s.own_begin, s.own_end, hay.size,
                                                 0, **flags)
                        m.count_records_device(p, c, counts.data_ptr())
                    assert bool((counts == want).all()), f"{kind} x{world} host={host} {flags}"
            m.set_pattern_ids(False)
        # world-1 gather with no_overlap, then the count on the root
        want = torch.from_numpy(_oracle_only(m, path, hay, sf, no_overlap=True).astype(np.int64)).cuda()
        m.set_pattern_ids(True)
        m.comm_init(Matcher.comm_unique_id(), 0, 1)
        cnt, ptr = m.match_shard(dev.data_ptr(), 0, hay.size, 0, hay.size, hay.size, 0)
        total, gptr = m.gather_records(ptr, cnt, 0, no_overlap=True)
        counts = torch.zeros(P, dtype=torch.int64, device="cuda")
        m.count_records_device(gptr, total, counts.data_ptr())
        assert bool((counts == want).all()) and total == int(want.sum().item())


def test_host_span_path_counts(store_cache, monkeypatch):
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    n = 9 * MIB + 12345
    hay = inputs.text_haystack(n, 7 + n)
    for edge in range(4 * MIB, n - 6, 4 * MIB):
        hay[edge - 5:edge + 6] = np.frombuffer(b"Christopher", dtype=np.uint8)
    hb = hay.tobytes()
    kws = ({}, {"longest_only": True, "no_overlap": True})
    for sf in ((0, 0, 0), (1, 1, 1)):
        path = store_cache("span-names", names, sf)
        with Matcher(path) as whole:
            wants = [_oracle_only(whole, path, hb, sf, **kw) for kw in kws]
        monkeypatch.setenv("OLM_HOST_SPAN_BYTES", str(4 * MIB))
        with Matcher(path) as m:
            for kw, want in zip(kws, wants):
                counts = np.zeros(m.pattern_count, dtype=np.uint64)
                total = _count_c(m, hb, counts, **kw)
                assert (counts == want).all() and total == int(want.sum()), f"{sf} {kw}"
                assert not m._match_records(hb[:MIB])["_pad"].any()  # ids stay off
        monkeypatch.delenv("OLM_HOST_SPAN_BYTES")


@pytest.mark.parametrize("sf", [(0, 0, 0), (1, 1, 1)])
def test_multi_matcher_counts(store_cache, sf):
    names = inputs.case_patterns(dict(patterns="names", store_flags=sf))
    path = store_cache("multi-names", names, sf)
    hay = inputs.text_haystack(13 * MIB + 4321, 31 + sum(sf)).tobytes()
    with Matcher(path) as one, Matcher(path, devices=_devices(2)) as many:
        for kw in ({}, {"no_overlap": True}, {"longest_only": True, "no_overlap": True}):
            want = _oracle_only(one, path, hay, sf, **kw)
            counts = np.zeros(many.pattern_count, dtype=np.uint64)
            total = _count_c(many, hay, counts, **kw)
            assert (counts == want).all() and total == int(want.sum()), f"{sf} {kw}"


def test_multi_matcher_counts_with_window_tails(store_cache):
    """A transforming store with 2..4 byte patterns under word_boundary runs on the first GPU alone."""
    sf = (1, 1, 1)
    pats = [b"ab", b"the", b"king", b"lord", b"of", b"and", b"jesus"]
    path = store_cache("counts-tails", b"\n".join(pats), sf)
    hay = inputs.text_haystack(9 * WINDOW + 77, 3).tobytes()
    with Matcher(path) as one, Matcher(path, devices=_devices(2)) as many:
        for kw in ({"word_boundary": True}, {"word_boundary": True, "longest_only": True, "no_overlap": True}):
            want = _oracle_only(one, path, hay, sf, **kw)
            assert want.sum() > 0
            assert (many.pattern_counts(hay, **kw) == want).all(), kw


# ---- errors ----------------------------------------------------------------------------------

def test_errors(store_cache, tmp_path):
    torch = pytest.importorskip("torch")
    path = store_cache("counts-skew", b"abcde\nzzzzzz\nab\nq\n")
    with Matcher(path) as m:
        P = m.pattern_count
        counts = torch.zeros(P, dtype=torch.int64, device="cuda")
        rec = torch.zeros((3, 3), dtype=torch.int64, device="cuda")
        rec[:, 1] = 5 | (torch.tensor([0, P, 1], device="cuda") << 32)
        with pytest.raises(RuntimeError):
            m.count_records_device(rec.data_ptr(), 3, counts.data_ptr())
        rec[1, 1] = 5 | ((P - 1) << 32)
        counts.zero_()
        m.count_records_device(rec.data_ptr(), 3, counts.data_ptr())
        assert counts.tolist() == [1, 1] + [0] * (P - 3) + [1]
        total = C.c_uint64()
        hay = b"abcde abcde"
        assert m._lib.olm_cuda_count_patterns(m._matcher, hay, len(hay), *([0] * 7), None, C.byref(total)) == -1
        assert m._lib.olm_cuda_count_patterns_device(m._matcher, counts.data_ptr(), 16, *([0] * 7), None,
                                                     C.byref(total)) == -1
        assert m._lib.olm_cuda_count_records(m._matcher, rec.data_ptr(), 3, None) == -1
    # a malformed store: the catalogue is refused, the count call fails without crashing
    ok = str(tmp_path / "ok.olm")
    Compiler.compile_from_buffer(ok, b"abcdefg\nabcdxyz1\nqwerty\nab\n")
    data = bytearray(open(ok, "rb").read())
    _, buckets = _bucket_records(bytes(data))
    two = next(b for b in buckets if len(b) == 2)
    data[two[1]:two[1] + 8] = data[two[0]:two[0] + 8]
    bad = str(tmp_path / "bad.olm")
    open(bad, "wb").write(bytes(data))
    with pytest.raises(RuntimeError):  # the matcher itself may refuse the file
        with Matcher(bad) as m:
            counts = np.zeros(8, dtype=np.uint64)
            total = C.c_uint64()
            hay = b"abcdefg qwerty"
            if m._lib.olm_cuda_count_patterns(m._matcher, hay, len(hay), *([0] * 7), counts.ctypes.data,
                                              C.byref(total)) != 0:
                raise RuntimeError("refused")
