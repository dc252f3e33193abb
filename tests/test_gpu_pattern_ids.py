"""Pattern ids (include/olm_b200.h "pattern ids"): the catalogue of a store and the id of each
record's pattern, resolved on the GPU -- needs a B200.

The id of a record is checked against the record's own source span: its bytes, normalised the way
the store normalises (without the trailing-space trim, which belongs to the end of a window, not to
a match), must be the bytes `Matcher.pattern(id)` returns.
"""
import random
import struct

import numpy as np
import pytest

import inputs
from conftest import describe_diff, same_matches
from omega_match_b200 import MATCH_IDS_DTYPE, Compiler, Matcher
from omega_match_b200.sharding import WINDOW, shard_plan
from oracle.oracle import Oracle
from test_gpu_multi import _devices
from test_gpu_parity import _colliding_patterns

pytestmark = pytest.mark.gpu

MIB = 1 << 20
EDGE_FLAGSETS = ({}, {"word_boundary": True}, {"longest_only": True, "no_overlap": True}, {"line_start": True},
                 {"line_end": True, "word_suffix": True}, {"word_prefix": True})


def _normalised_span(span: bytes, sf) -> bytes:
    """What the store keeps of a matched source span: transform_apply without the final trim."""
    return Oracle.transform(span + b"Q", *sf)[0][:-1] if any(sf) else span


def _check_ids(m: Matcher, hay: bytes, got: np.ndarray, sf, what=""):
    cat = {}
    norm = {}
    n = m.pattern_count
    for off, ln, pid in zip(got["offset"].tolist(), got["len"].tolist(), got["pattern_id"].tolist()):
        assert pid < n, f"{what}: record ({off}, {ln}) has id {pid:#x} (catalogue of {n})"
        span = bytes(hay[off:off + ln])
        if span not in norm:
            norm[span] = _normalised_span(span, sf)
        if pid not in cat:
            cat[pid] = m.pattern(pid)
        assert cat[pid] == norm[span], f"{what}: record ({off}, {ln}) {span!r} -> id {pid} = {cat[pid]!r}"


def _check_call(m: Matcher, o: Oracle, hay, sf, **flags):
    """match_ids: the oracle's stream, the stream of a call without ids, and a right id on every record."""
    hay = bytes(hay)
    got = m.match_ids(hay, **flags)
    assert got.dtype == MATCH_IDS_DTYPE
    want = o.match(hay, **flags)
    assert same_matches(got, want), f"{sf} {flags}: " + describe_diff(got, want)
    plain = m._match_records(hay, **flags)  # ids off
    assert same_matches(got, plain)
    assert not plain["_pad"].any(), "ids off: the pad bytes must stay 0"
    _check_ids(m, hay, got, sf, f"{sf} {flags}")
    return got


# ---- the catalogue ---------------------------------------------------------------------------

CATALOGUE_LINES = [b"Hello", b"hello", b"HEL-LO", b"he llo", b"he  llo", b"x", b"X", b"ab", b"AB", b"a-b", b"ab",
                   b"abc", b"ABC", b"abcd", b"a.bcd", b"zz top", b"ZZ  TOP", b"Zz top!", b"o-malley", b"OMALLEY",
                   b"O'Malley", b"q" * 30, b"Q" * 30, b"abcdefghijklmnopqrstuvwxyz0123", b"the", b"The", b"t-h-e",
                   b"Hello", b"hello world", b"HELLO, WORLD", b"9", b"99", b"999", b"9999", b"99999", b"abcdefg"]


@pytest.mark.parametrize("sf", [(0, 0, 0), (1, 0, 0), (1, 1, 1)])
def test_catalogue_order_and_bytes(store_cache, tmp_path, sf):
    lines = [p for p in CATALOGUE_LINES if inputs.py_normalize(p, *sf)]
    buf = b"\n".join(lines) + b"\n"
    path = store_cache("ids-catalogue", buf, sf)
    st = Compiler.compile_from_buffer(str(tmp_path / "stats.olm"), buf, *map(bool, sf))
    norm = [Oracle.transform(p, *sf)[0] if any(sf) else p for p in lines]
    longs = list(dict.fromkeys(p for p in norm if len(p) >= 5))  # first appearance
    shorts = sorted(set(p for p in norm if len(p) < 5), key=lambda p: (len(p), p))
    with Matcher(path) as m:
        assert m.pattern_count == st.stored_pattern_count + st.short_pattern_count == len(longs) + len(shorts)
        assert [m.pattern(i) for i in range(m.pattern_count)] == longs + shorts
        with pytest.raises(IndexError):
            m.pattern(m.pattern_count)
        with pytest.raises(IndexError):
            m.pattern(-1)


# ---- ids per record --------------------------------------------------------------------------

@pytest.mark.parametrize("sf", inputs.STORE_FLAG_SETS)
def test_ids_on_edge_haystacks(store_cache, sf):
    from test_gpu_parity import EDGE_PATTERNS
    buf = b"\n".join(p for p in EDGE_PATTERNS if inputs.py_normalize(p, *sf)) + b"\n"
    path = store_cache("edge", buf, sf)
    o = Oracle.from_olm(path)
    hays = [b"", b"a", b"abcd", b"abcde", b"xabcdefghij", b"abcdefghij" * 3, b"x" * 41, b"x" * 450,
            b"hello world", b"Hello,  World!\n", b"the King\nline\n", b"abcd" * 1000, (b"abcde " * 7000)[:32768 + 5],
            b"q" * 32766 + b"abcdefghij", b"q" * 32760 + b"x" * 220, b"A-b-C-d-E, h.e.l.l.o \t\t w-o-r-l-d"]
    with Matcher(path) as m:
        for hay in hays:
            for flags in EDGE_FLAGSETS:
                _check_call(m, o, hay, sf, **flags)


@pytest.mark.parametrize("seed", range(6))
def test_ids_on_random_stores_and_haystacks(store_cache, seed):
    rng = random.Random(7000 + seed)
    alph = b"abcABC xyz.,-'\n\t_09"
    pats = set()
    while len(pats) < rng.choice([5, 40, 400]):
        pats.add(bytes(rng.choice(b"abcABC xyz.-'_09") for _ in range(rng.choice([1, 2, 2, 3, 3, 4, 4, 5, 6, 9, 14, 30]))))
    sf = inputs.STORE_FLAG_SETS[seed % len(inputs.STORE_FLAG_SETS)]
    lines = sorted(p for p in pats if inputs.py_normalize(p, *sf))
    lines += lines[::3]  # duplicates
    path = store_cache(f"ids-fuzz{seed}", b"\n".join(lines), sf)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        for i in range(8):
            n = rng.choice([0, 1, 5, 300, 4000, 40000, 70001])
            hay = bytes(rng.choice(alph) for _ in range(n))
            _check_call(m, o, hay, sf, **EDGE_FLAGSETS[i % len(EDGE_FLAGSETS)])


def test_ids_of_short_patterns_and_grams(store_cache):
    """1..4 byte patterns, 4-byte patterns that are also the key grams of long patterns."""
    pats = [b"a", b"b", b"ab", b"ba", b"abc", b"bca", b"abcd", b"bcda", b"abcdef", b"abcdxyz", b"bcdab", b"cdab"]
    for sf in ((0, 0, 0), (1, 0, 0), (1, 1, 1)):
        path = store_cache("ids-short", b"\n".join(pats), sf)
        o = Oracle.from_olm(path)
        rng = random.Random(3)
        hay = bytes(rng.choice(b"abcdABCD xyz-") for _ in range(50000))
        with Matcher(path) as m:
            for flags in EDGE_FLAGSETS:
                _check_call(m, o, hay, sf, **flags)


@pytest.mark.parametrize("k", [5, 6, 7, 8])
def test_ids_of_colliding_keys(store_cache, k):
    a, b = _colliding_patterns(k)
    path = store_cache(f"ids-collide{k}", a + b"\n" + b + b"\n")
    o = Oracle.from_olm(path)
    hay = b"..." + a + b" " + b + b"|" + b + a + b"\n" + a[:k] + b[k:] + b"|" + b[:k] + a[k:]
    with Matcher(path) as m:
        got = _check_call(m, o, hay, (0, 0, 0))
        assert sorted(set(got["pattern_id"].tolist())) == [0, 1]


def test_ids_of_long_patterns_across_tiles(store_cache):
    rng = np.random.default_rng(5)
    pats = [bytes(rng.integers(97, 123, size=n, dtype=np.uint8)) for n in (5, 8, 9, 16, 100, 113, 114, 500, 5000)]
    path = store_cache("longpats", b"\n".join(pats))
    o = Oracle.from_olm(path)
    hay = bytearray(rng.integers(97, 123, size=200_000, dtype=np.uint8).tobytes())
    for i, p in enumerate(pats):
        for at in (32768 - len(p) // 2, 65536 - 3, 100_000 + 37 * i, 200_000 - len(p)):
            if at >= 0:
                hay[at:at + len(p)] = p
    with Matcher(path) as m:
        for flags in ({}, {"word_boundary": True}, {"longest_only": True, "no_overlap": True}):
            _check_call(m, o, hay, (0, 0, 0), **flags)


def test_ids_across_window_edges(store_cache):
    """4 MiB window edges of normalising stores, and a stored pattern that still ends in a space."""
    W = WINDOW
    hay = bytearray(b"." * (W + 100))
    hay[W - 5:W + 5] = b"helloworld"
    hay[W + 20:W + 40] = b"Hel-lo, wor ld ab  x"
    for sf in ((1, 0, 0), (1, 1, 0), (1, 1, 1), (0, 1, 0), (0, 0, 1)):
        pats = [p for p in (b"HELLOWORLD", b"hello", b"hel lo", b"ab  ", b"ab", b"zq") if inputs.py_normalize(p, *sf)]
        path = store_cache("ids-window", b"\n".join(pats), sf)
        o = Oracle.from_olm(path)
        with Matcher(path) as m:
            for flags in ({}, {"word_boundary": True}, {"longest_only": True, "no_overlap": True}):
                _check_call(m, o, hay, sf, **flags)


def test_id_of_a_pattern_that_ends_in_a_space(store_cache):
    """Ignore-case only: `ab  ` is stored as `AB ` (one trailing space trimmed); a match of it in the
    middle of a window keeps its space and must resolve to `AB `, not to `AB` or to nothing."""
    sf = (1, 0, 0)
    path = store_cache("ids-space", b"ab  \nab\nx\n", sf)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        assert sorted(m.pattern(i) for i in range(m.pattern_count)) == [b"AB", b"AB ", b"X"]
        got = _check_call(m, o, b"zz ab  yy Ab x aB ", sf)
        names = [(int(a), m.pattern(int(i))) for a, i in zip(got["offset"], got["pattern_id"])]
        assert (3, b"AB ") in names and (3, b"AB") in names


# ---- nothing else changes --------------------------------------------------------------------

def test_switching_ids_off_restores_zero_pads(store_cache):
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    path = store_cache("ids-names", names, (0, 0, 0))
    hay = inputs.text_haystack(3 * MIB + 7, 5)
    with Matcher(path) as m:
        before = m._match_records(hay)
        assert not before["_pad"].any()
        m.set_pattern_ids(True)
        on = m._match_records(hay)
        assert on.size and (on["offset"] == before["offset"]).all() and (on["len"] == before["len"]).all()
        assert (on["match"] == before["match"]).all()
        assert on["_pad"].max() < m.pattern_count
        m.set_pattern_ids(False)
        after = m._match_records(hay)
        assert after.tobytes() == before.tobytes()
        ids = m.match_ids(hay)  # switches on for one call only
        assert (ids["pattern_id"] == on["_pad"]).all()
        assert not m._match_records(hay)["_pad"].any()


# ---- every path carries ids ------------------------------------------------------------------

def _device_ids(torch, ptr, count):
    from test_gpu_parity import _device_records
    rec = _device_records(torch, ptr, count)
    a = rec.cpu().numpy()
    out = np.zeros(a.shape[0], dtype=MATCH_IDS_DTYPE)
    out["offset"] = a[:, 0].astype(np.uint64)
    out["len"] = (a[:, 1] & 0xFFFFFFFF).astype(np.uint32)
    out["pattern_id"] = ((a[:, 1] >> 32) & 0xFFFFFFFF).astype(np.uint32)
    return out, rec


@pytest.mark.parametrize("kind", ["plain", "windowed"])
def test_device_shard_sort_and_gather_paths(store_cache, kind):
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
    hb = hay.tobytes()
    dev = torch.zeros(hay.size + 64, dtype=torch.uint8, device="cuda")
    dev[:hay.size] = torch.from_numpy(hay).cuda()
    torch.cuda.synchronize()
    with Matcher(path) as m:
        for flags in ({}, {"longest_only": True, "word_boundary": True}, {"no_overlap": True, "longest_only": True}):
            want = m.match_ids(hb, **flags)  # the host entry point
            _check_ids(m, hb, want, sf, f"{kind} host {flags}")
            m.set_pattern_ids(True)
            cnt, ptr = m.match_device(dev.data_ptr(), hay.size, **flags)
            got, rec = _device_ids(torch, ptr, cnt)
            assert got.tobytes() == want.tobytes(), f"{kind} device {flags}"
            assert bool((rec[:, 2] == rec[:, 0] + dev.data_ptr()).all())
            if not flags:  # the radix sort moves ids with their records
                perm = torch.randperm(cnt, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
                shuffled = rec[perm].contiguous()
                m.sort_records_device(shuffled.data_ptr(), cnt)
                assert bool((shuffled == rec).all())
            fl = {k: v for k, v in flags.items() if k != "no_overlap"}
            for world in (2, 4):
                for host in (False, True):
                    parts = []
                    for s in shard_plan(hay.size, world, largest, windowed=any(sf)):
                        ln = s.slice_end - s.slice_begin
                        if host:
                            hslice = np.ascontiguousarray(hay[s.slice_begin:s.slice_end])
                            c, p = m.match_shard_host(hslice.ctypes.data, s.slice_begin, ln, s.own_begin, s.own_end,
                                                      hay.size, 0, **fl)
                        else:
                            sl = torch.zeros(((ln + 15) // 16) * 16 + 16, dtype=torch.uint8, device="cuda")
                            sl[:ln] = dev[s.slice_begin:s.slice_end]
                            torch.cuda.synchronize()
                            c, p = m.match_shard(sl.data_ptr(), s.slice_begin, ln, s.own_begin, s.own_end, hay.size,
                                                 0, **fl)
                        parts.append(_device_ids(torch, p, c)[1].clone())
                    allrec = torch.cat(parts).contiguous()
                    n = allrec.shape[0]
                    if flags.get("no_overlap"):
                        n = m.no_overlap_device(allrec.data_ptr(), n)
                    a = allrec[:n].cpu().numpy()
                    got = np.zeros(n, dtype=MATCH_IDS_DTYPE)
                    got["offset"], got["len"] = a[:, 0], a[:, 1] & 0xFFFFFFFF
                    got["pattern_id"] = (a[:, 1] >> 32) & 0xFFFFFFFF
                    assert got.tobytes() == want.tobytes(), f"{kind} x{world} host={host} {flags}"
            m.set_pattern_ids(False)
        # the library's gather with a world of one keeps whole records
        m.set_pattern_ids(True)
        m.comm_init(Matcher.comm_unique_id(), 0, 1)
        cnt, ptr = m.match_shard(dev.data_ptr(), 0, hay.size, 0, hay.size, hay.size, 0)
        total, gptr = m.gather_records(ptr, cnt, 0, no_overlap=True)
        got, _ = _device_ids(torch, gptr, total)
        want = m.match_ids(hb, no_overlap=True)
        assert got.tobytes() == want.tobytes()


def test_host_span_path_carries_ids(store_cache, monkeypatch):
    names = inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0)))
    n = 9 * MIB + 12345
    hay = inputs.text_haystack(n, 7 + n)
    for edge in range(4 * MIB, n - 6, 4 * MIB):
        hay[edge - 5:edge + 6] = np.frombuffer(b"Christopher", dtype=np.uint8)
    hb = hay.tobytes()
    for sf in ((0, 0, 0), (1, 1, 1)):
        path = store_cache("span-names", names, sf)
        with Matcher(path) as whole:
            wants = [whole.match_ids(hb, **kw) for kw in ({}, {"longest_only": True, "no_overlap": True})]
        monkeypatch.setenv("OLM_HOST_SPAN_BYTES", str(4 * MIB))
        with Matcher(path) as m:
            for kw, want in zip(({}, {"longest_only": True, "no_overlap": True}), wants):
                got = m.match_ids(hb, **kw)
                assert got.tobytes() == want.tobytes(), f"{sf} {kw}"
                _check_ids(m, hb, got, sf, f"spans {sf} {kw}")
        monkeypatch.delenv("OLM_HOST_SPAN_BYTES")


@pytest.mark.parametrize("sf", [(0, 0, 0), (1, 1, 1)])
def test_multi_matcher_carries_ids(store_cache, sf):
    names = inputs.case_patterns(dict(patterns="names", store_flags=sf))
    path = store_cache("multi-names", names, sf)
    hay = inputs.text_haystack(13 * MIB + 4321, 31 + sum(sf)).tobytes()
    with Matcher(path) as one, Matcher(path, devices=_devices(2)) as many:
        for kw in ({}, {"no_overlap": True}, {"longest_only": True, "no_overlap": True}):
            want = one.match_ids(hay, **kw)
            assert many.match_ids(hay, **kw).tobytes() == want.tobytes(), f"{sf} {kw}"


# ---- at scale --------------------------------------------------------------------------------

def test_ids_at_one_million_patterns(store_cache):
    """256 MiB of the cfg5 haystack x 1 M patterns: every planted pattern's record carries that
    pattern's id (all patterns are long and distinct: id = index in the compile input)."""
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
    # where inputs.plant puts them: one pattern per 4 KiB block
    nb = n // 4096
    r = inputs.rand_u64(inputs.SEED_H5 ^ 0x77, nb, 0)
    r2 = inputs.rand_u64((inputs.SEED_H5 ^ 0x77) ^ 0x5555, nb, 0)
    idx = (r2 % np.uint64(len(pats))).astype(np.int64)
    lens = np.array([len(pats[i]) for i in idx], dtype=np.int64)
    at = np.arange(nb, dtype=np.int64) * 4096 + 1 + (r % (4096 - 2 - lens).astype(np.uint64)).astype(np.int64)
    with Matcher(path) as m:
        assert m.pattern_count == len(pats)
        m.set_pattern_ids(True)
        cnt, ptr = m.match_device(hay.data_ptr(), n)
        got, _ = _device_ids(torch, ptr, cnt)
        t = m.last_timing()
        assert t["total_ms"] >= t["scan_ms"]
        rid = {(int(o), int(ln)): int(i) for o, ln, i in zip(got["offset"], got["len"], got["pattern_id"])}
        for a, ln, i in zip(at.tolist(), lens.tolist(), idx.tolist()):
            assert rid.get((a, ln)) == i, f"planted pattern {i} at {a}"
        host = hay[:n].cpu().numpy()
        sample = np.random.default_rng(11).choice(cnt, size=min(cnt, 100_000), replace=False)
        for k in sample.tolist():
            o, ln, i = int(got["offset"][k]), int(got["len"][k]), int(got["pattern_id"][k])
            assert pats[i] == host[o:o + ln].tobytes() == m.pattern(i)


# ---- errors ----------------------------------------------------------------------------------

def _bucket_records(data: bytes):
    """File offsets of the {u64 store_off, u32 len} bucket records of a store, grouped by bucket."""
    store_bytes, = struct.unpack_from("<Q", data, 16)
    bloom_bytes, blob_bytes, table_size = struct.unpack_from("<III", data, 36)
    p = 72 + store_bytes + 12 + bloom_bytes + 8 + 4 * table_size
    end, buckets = p + blob_bytes, []
    while p < end:
        count, = struct.unpack_from("<I", data, p + 4)
        buckets.append([p + 8 + 16 * j for j in range(count)])
        p += 8 + 16 * count
    return store_bytes, buckets


@pytest.mark.parametrize("damage", ["duplicate-offset", "offset-out-of-range"])
def test_malformed_catalogue_is_rejected(tmp_path, damage):
    path = str(tmp_path / "ok.olm")
    Compiler.compile_from_buffer(path, b"abcdefg\nabcdxyz1\nqwerty\nab\n")
    data = bytearray(open(path, "rb").read())
    store_bytes, buckets = _bucket_records(bytes(data))
    two = next(b for b in buckets if len(b) == 2)
    if damage == "duplicate-offset":
        data[two[1]:two[1] + 8] = data[two[0]:two[0] + 8]
    else:
        struct.pack_into("<Q", data, two[1], store_bytes)
    bad = str(tmp_path / f"{damage}.olm")
    open(bad, "wb").write(bytes(data))
    with pytest.raises(RuntimeError):  # the matcher itself may refuse the file; ids must never crash
        with Matcher(bad) as m:
            m.set_pattern_ids(True)
    with Matcher(path) as m:  # the intact store
        m.set_pattern_ids(True)
        assert m.pattern_count == 4
