"""Match streams (include/olm_b200.h "Streams"): pieces pushed one after another return, concatenated,
the records of one call over the concatenation -- host pieces, device pieces and a mix, cut anywhere."""
import ctypes as C
import os

import numpy as np
import pytest

import inputs
from conftest import describe_diff, same_matches
from omega_match_b200 import Matcher, _lib
from oracle.oracle import Oracle
from test_gpu_parity import _device_records

pytestmark = pytest.mark.gpu

W = inputs.WINDOW
FLAGS = ("no_overlap", "longest_only", "word_boundary", "word_prefix", "word_suffix", "line_start", "line_end")


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def store_largest(path) -> int:
    info = _lib.StoreInfoC()
    assert _lib.load().olm_store_inspect(os.fsencode(path), C.byref(info)) == 0
    return int(info.largest)


def expected_settled(prev, received, largest, windowed, last):
    if last:
        return received
    if windowed:
        return received // W * W
    k = received - largest - 1 if received > largest + 1 else 0
    return max(prev, k if k >= 16 else 0)


def stream_records(m, hay: bytes, cuts, kinds, torch=None, largest=None, windowed=False, misalign=False, **flags):
    """Push hay cut at `cuts` ("h": host piece, "d": device piece) -> the concatenated records; checks
    received / settled after every push when `largest` is given."""
    edges = [0] + sorted(cuts) + [len(hay)]
    got, settled = [], 0
    with m.stream(**flags) as s:
        for i in range(len(edges) - 1):
            piece, last = hay[edges[i]:edges[i + 1]], i == len(edges) - 2
            if kinds[i % len(kinds)] == "h":
                r = s.push(piece, last=last)
                got.append(np.array(list(zip(r["offset"].tolist(), r["len"].tolist())), dtype=np.uint64).reshape(-1, 2))
            else:
                off = 1 if misalign and i % 3 == 1 else 0  # an unaligned device piece is copied, not scanned in place
                buf = torch.zeros(len(piece) + 32, dtype=torch.uint8, device="cuda")
                if piece:
                    buf[off:off + len(piece)] = torch.frombuffer(bytearray(piece), dtype=torch.uint8).cuda()
                ptr, cnt = s.push_device(buf.data_ptr() + off, len(piece), last=last)
                a = _device_records(torch, ptr, cnt).cpu().numpy()
                buf.fill_(0x2e)  # the caller reuses its buffer right away
                got.append(np.stack([a[:, 0], a[:, 1] & 0xFFFFFFFF], axis=1).astype(np.uint64) if cnt else np.zeros((0, 2), np.uint64))
            if largest is not None:
                settled = expected_settled(settled, edges[i + 1], largest, windowed, last)
                assert (s.received, s.settled) == (edges[i + 1], settled)
    a = np.concatenate(got) if got else np.zeros((0, 2), np.uint64)
    out = np.zeros(a.shape[0], dtype=[("offset", "<u8"), ("len", "<u4")])
    out["offset"] = a[:, 0]
    out["len"] = a[:, 1]
    return out


def check_stream(m, o, hay, cuts, kinds, torch=None, **flags):
    got = stream_records(m, hay, cuts, kinds, torch, **flags)
    want = o.match(hay, **{k: v for k, v in flags.items() if k in FLAGS})
    assert same_matches(got, want), f"{flags} cuts {sorted(cuts)[:8]} {kinds}: " + describe_diff(got, want)
    return got


def random_cuts(rng, n, k):
    cuts = set(int(c) for c in rng.integers(0, n + 1, size=k))
    cuts |= {c for c in (1, 2, n - 1) if 0 < c < n}
    return sorted(cuts)


@pytest.mark.parametrize("seed", range(6))
def test_random_cuts(store_cache, torch, seed):
    """Random stores of every pattern length under every store flag set, random match flags, haystacks cut
    at random (empty and 1-byte pieces, inside matches, between '\\r' and '\\n') into host pieces, device
    pieces and a mix."""
    import random
    rng = random.Random(3000 + seed)
    nrng = np.random.default_rng(seed)
    sf = inputs.STORE_FLAG_SETS[seed]
    pats = set()
    while len(pats) < rng.choice([3, 30, 300]):
        pats.add(bytes(rng.choice(b"abcABC xyz.-'_09") for _ in range(rng.choice([1, 2, 3, 4, 5, 6, 9, 12, 40]))))
    buf = b"\n".join(sorted(p for p in pats if inputs.py_normalize(p, *sf)))
    path = store_cache(f"stream-fuzz{seed}", buf, sf)
    o = Oracle.from_olm(path)
    with Matcher(path) as m:
        largest = store_largest(path)
        for rnd in range(6):
            n = rng.choice([0, 1, 5, 300, 4000, 70001])
            hay = bytes(rng.choice(b"abcABC xyz.,-'\n\r\r\n\t_09") for _ in range(n))
            kw = {f: rng.random() < 0.3 for f in FLAGS}
            cuts = random_cuts(nrng, n, rng.choice([1, 3, 20]))
            cuts += [i + 1 for i in range(n - 1) if hay[i:i + 2] == b"\r\n"][:3]  # inside "\r\n"
            cuts += cuts[:2]  # empty pieces
            for kinds in ("h", "d", "hd"):
                check_stream(m, o, hay, cuts, kinds, torch, misalign=rnd % 2 == 1, **kw)
            stream_records(m, hay, cuts, "dh", torch, largest=largest if not any(sf) else None, **kw)


@pytest.mark.parametrize("sf", [(1, 0, 0), (1, 1, 1)])
def test_window_edges(store_cache, torch, sf):
    """Case-folding and normalising stores with 2..4 byte patterns over 3+ windows, cut at every window
    edge -1, 0, +1 and mid-window; the stale-tail cases of the whole-call tests, cut into pieces."""
    path = store_cache("stream-win", b"ab\nzq\nhello\nabc\nHELLOWORLD\n", sf)
    o = Oracle.from_olm(path)
    rng = np.random.default_rng(11)
    hay = bytearray(rng.choice(np.frombuffer(b"abQz ,.hel\n", dtype=np.uint8), size=3 * W + 5000).tobytes())
    hay[W - 5:W + 5] = b"helloworld"
    hay[2 * W - 2:2 * W] = b"zq"
    hay[-2:] = b"ab"
    hay = bytes(hay)
    edge_cuts = sorted({w * W + d for w in (1, 2, 3) for d in (-1, 0, 1)} | {W // 2, 2 * W + 12345})
    with Matcher(path) as m:
        for flags in ({}, {"word_boundary": True}):
            for kinds in ("h", "d", "hd"):
                got = check_stream(m, o, hay, edge_cuts, kinds, torch, largest=None, **flags)
                assert got.size > 1000
            stream_records(m, hay, edge_cuts, "dh", torch, largest=store_largest(path), windowed=True, **flags)
        # test_window_edges_and_stale_tail: what window 0 leaves at scratch index 99 decides window 1
        hay2 = bytearray(b"." * W + b"y" * 96 + b" ab")
        for q in (False, True):
            if q:
                hay2[99] = ord("Q")
            want = o.match(bytes(hay2), word_boundary=True)
            for cuts in ([W], [W - 1, W + 50], [100, W + 1]):
                got = stream_records(m, bytes(hay2), cuts, "hd", torch, word_boundary=True)
                o.match(bytes(hay2), word_boundary=True)  # keep the oracle's scratch buffer in step
                assert same_matches(got, want), describe_diff(got, want)
        # test_stale_tail_across_calls_of_a_normalising_store: streams after a longer call
        for rnd in range(3):
            long_hay = bytes(rng.choice(np.frombuffer(b"abQz  ..,-q\n", dtype=np.uint8), size=int(rng.integers(3000, 9000))))
            check_stream(m, o, long_hay, random_cuts(rng, len(long_hay), 4), "hd", torch, word_boundary=True)
            for cut in rng.integers(5, 2500, size=3):
                short = long_hay[:int(cut)].rstrip(b" .,-\n") + b".ab"
                check_stream(m, o, short, random_cuts(rng, len(short), 3), "dh", torch, word_boundary=True)


def test_no_overlap_across_pushes(store_cache, torch):
    """A 250-byte pattern pushed in 1-byte pieces: a kept match that straddles a push edge drops the
    overlapping matches of the pieces after it; longest_only + no_overlap; line_end at the stream's end."""
    long_p = b"ab" * 125
    path = store_cache("stream-long", b"\n".join([long_p, b"ab" * 10, b"ba" * 7, b"b"]), (0, 0, 0))
    o = Oracle.from_olm(path)
    hay = b"x" + b"ab" * 400 + b"\nab"
    one_byte = list(range(1, len(hay)))
    with Matcher(path) as m:
        for flags in ({"no_overlap": True}, {"no_overlap": True, "longest_only": True}, {"line_end": True},
                      {"line_end": True, "no_overlap": True}):
            check_stream(m, o, hay, one_byte, "h", torch, largest=store_largest(path), **flags)
            check_stream(m, o, hay, one_byte[::7], "hdd", torch, **flags)
        got = check_stream(m, o, hay, list(range(5, len(hay), 97)), "d", torch, no_overlap=True)
        assert got.size > 3 and int(got["len"][0]) == len(long_p)


def test_settled_and_errors(store_cache, torch):
    path = store_cache("stream-small", b"hello\nab\nworld", (0, 0, 0))
    with Matcher(path) as m:
        with m.stream() as s:
            assert s.push(b"", last=True).size == 0
            assert (s.received, s.settled) == (0, 0)
            with pytest.raises(RuntimeError):
                s.push(b"hello")
        with m.stream() as s:
            r = s.push(b"hello world ab " * 3)
            assert s.received == 45 and s.settled == 45 - 6
            r2 = s.push(b"", last=True)
            assert s.settled == 45
            assert np.concatenate([r, r2])["offset"].tolist() == m.match_arrays(b"hello world ab " * 3)["offset"].tolist()
            with pytest.raises(RuntimeError):
                s.push(b"x", last=True)
        s = m.stream()
        s.close()
        with pytest.raises(RuntimeError):
            s.push(b"x")


def test_ids_and_counts(store_cache, torch):
    pats = [p for p in inputs.case_patterns(dict(patterns="names", store_flags=(0, 0, 0))).split(b"\n") if p]
    path = store_cache("stream-names", b"\n".join(pats), (0, 0, 0))
    hay = inputs.text_haystack(3 << 20, 5).tobytes()
    rng = np.random.default_rng(5)
    cuts = random_cuts(rng, len(hay), 9)
    edges = [0] + cuts + [len(hay)]
    with Matcher(path) as m:
        for flags in ({}, {"no_overlap": True}, {"longest_only": True, "word_boundary": True}):
            want = m.match_ids(hay, **flags)
            m.set_pattern_ids(True)
            with m.stream(**flags) as s:
                got = np.concatenate([s.push(hay[a:b], last=b == len(hay)) for a, b in zip(edges, edges[1:])])
            with m.stream(**flags) as s:  # device pieces: the pads hold the ids
                parts = []
                for a, b in zip(edges, edges[1:]):
                    t = torch.frombuffer(bytearray(hay[a:b]) or bytearray(1), dtype=torch.uint8).cuda()
                    ptr, cnt = s.push_device(t.data_ptr(), b - a, last=b == len(hay))
                    parts.append(_device_records(torch, ptr, cnt).cpu().numpy())
                dev = np.concatenate(parts)
            m.set_pattern_ids(False)
            assert got.dtype.names == ("offset", "len", "pattern_id")
            assert np.array_equal(got, want)
            assert np.array_equal(dev[:, 0].astype(np.uint64), want["offset"])
            assert np.array_equal((dev[:, 1] >> 32).astype(np.uint32), want["pattern_id"])
            whole = m.pattern_counts(hay, **flags)
            for mix in (False, True):  # count pushes alone, and mixed with record pushes (ids on)
                counts = np.zeros(m.pattern_count, dtype=np.uint64)
                total = 0
                m.set_pattern_ids(mix)
                with m.stream(**flags) as s:
                    for i, (a, b) in enumerate(zip(edges, edges[1:])):
                        if mix and i % 2:
                            r = s.push(hay[a:b], last=b == len(hay))
                            np.add.at(counts, r["pattern_id"].astype(np.int64), np.uint64(1))
                            total += r.size
                        else:
                            total += s.count(hay[a:b], counts, last=b == len(hay))
                m.set_pattern_ids(False)
                assert total == want.size
                assert np.array_equal(counts, whole)


@pytest.mark.parametrize("sf", [(0, 0, 0), (1, 1, 1)])
def test_exact_statistics_sum_to_one_call(store_cache, torch, sf):
    path = store_cache("stream-stats", b"hello\nab\nworld wide\nzq\nabcdefgh", sf)
    hay = inputs.text_haystack(W + 300_000, 9).tobytes()
    cuts = [1000, W - 1, W + 7, W + 200_000]
    with Matcher(path) as m:
        m.set_exact_stats(True)
        for kinds in ("h", "d"):
            m.reset_match_stats()
            m.match_arrays(hay, word_boundary=True)
            one = m.get_match_stats()
            m.reset_match_stats()
            stream_records(m, hay, cuts, kinds, torch, word_boundary=True)
            assert m.get_match_stats() == one


def test_past_4gib_in_device_pieces(store_cache, torch):
    """About 5 GiB of cfg4's synthetic haystack on the device in 512 MiB pieces: equal to one
    match_device over the whole buffer, offsets above 2^32 included; record.match = base + offset."""
    import synth_torch
    pats = list(inputs._pattern_set("tlds")) + inputs.synth_short_patterns()
    path = store_cache("stream-cfg4", b"\n".join(pats), (0, 0, 0))
    n = 5 << 30
    piece = 512 << 20
    hay = synth_torch.synth_haystack_torch(n + 64, inputs.SEED_H4, device="cuda")
    base = 1 << 40
    with Matcher(path) as m:
        cnt, ptr = m.match_device(hay.data_ptr(), n, match_ptr_base=base)
        whole = _device_records(torch, ptr, cnt)
        at = 0
        with m.stream(match_ptr_base=base) as s:
            for b in range(0, n, piece):
                ptr, c = s.push_device(hay.data_ptr() + b, min(piece, n - b), last=b + piece >= n)
                part = _device_records(torch, ptr, c)
                assert torch.equal(part, whole[at:at + c])
                at += c
        assert at == cnt and int(whole[-1, 0]) > (1 << 32)
        assert bool((whole[:, 2] == whole[:, 0] + base).all())


def test_buffer_reuse_and_interleaved_streams(store_cache, torch):
    path = store_cache("stream-two", b"hello\nab\nworld\nlong pattern here", (0, 0, 0))
    o = Oracle.from_olm(path)
    rng = np.random.default_rng(3)
    hays = [bytes(rng.choice(np.frombuffer(b"helloab world long pattern here\n", dtype=np.uint8), size=200_000))
            for _ in range(2)]
    cuts = [sorted(rng.integers(1, 200_000, size=12).tolist()) for _ in range(2)]
    bases = [0x1000, 0x7000_0000_0000]
    with Matcher(path) as m:
        streams = [m.stream(match_ptr_base=bases[k], no_overlap=True) for k in range(2)]
        buf = torch.empty(200_032, dtype=torch.uint8, device="cuda")  # one device buffer, reused by both
        got = [[], []]
        edges = [[0] + c + [200_000] for c in cuts]
        for i in range(len(edges[0]) - 1):
            for k in range(2):
                a, b = edges[k][i], edges[k][i + 1]
                buf[:b - a] = torch.frombuffer(bytearray(hays[k][a:b]) or bytearray(1), dtype=torch.uint8).cuda()[:b - a]
                ptr, cnt = streams[k].push_device(buf.data_ptr(), b - a, last=i == len(edges[k]) - 2)
                r = _device_records(torch, ptr, cnt).cpu().numpy()
                buf.fill_(ord("a"))
                assert (r[:, 2] == r[:, 0] + bases[k]).all()
                got[k].append(r)
        for k in range(2):
            streams[k].close()
            r = np.concatenate(got[k])
            mm = np.zeros(r.shape[0], dtype=[("offset", "<u8"), ("len", "<u4")])
            mm["offset"], mm["len"] = r[:, 0], r[:, 1] & 0xFFFFFFFF
            want = o.match(hays[k], no_overlap=True)
            assert same_matches(mm, want), describe_diff(mm, want)
