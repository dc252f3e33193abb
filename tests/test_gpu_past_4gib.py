"""A whole call on a haystack above 2^32, record for record -- needs a B200 with 40 GiB free.

No oracle runs on 4 GiB, but a periodic haystack needs none.  B is one transform window (4 MiB): 64
'0' bytes, 512 KiB of text (inputs.text_haystack), '0' bytes up to its last byte, which is '\\n'.  No
pattern of the store holds a '0', so no match touches a copy boundary, no predicate reads across one, no
window ends in a match (stale tails stay out of it) and every line ends inside its copy.  (The '0' run
keeps 1 100 copies at a few GiB of records.)  H is B repeated 1 100 times: 4.3 GiB, and the copies from
1 024 on lie wholly above 2^32.  Every result on H is then copy 0's result shifted copy by copy: the
records, the pattern ids and counts, the line positions, the matching lines and the listing.
"""
import time

import numpy as np
import pytest

import inputs
from omega_match_b200 import Matcher
from oracle.oracle import Oracle
from test_gpu_lines import _rle
from test_gpu_parity import _as_matches, _device_records, _DevBytes
from test_lines_cpu import positions

pytestmark = pytest.mark.gpu

W = inputs.WINDOW
K = 1100
TEXT = 512 * 1024
STORES = {(0, 0, 0): "ids-names", (1, 1, 1): "counts-names-111"}
FLAG_SETS = [{}, {"word_boundary": True}, {"longest_only": True, "no_overlap": True}]


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def periodic(torch):
    """(B on the host, H on the device, a record of the peak device memory in use)"""
    t0 = time.perf_counter()
    torch.cuda.empty_cache()
    if torch.cuda.mem_get_info()[0] < 40 << 30:
        pytest.skip("needs 40 GiB of free device memory")
    b = np.full(W, ord("0"), dtype=np.uint8)
    b[64:64 + TEXT] = inputs.text_haystack(TEXT, 0x4B1D)
    b[-1] = 10
    h = torch.zeros(K * W + 4096, dtype=torch.uint8, device="cuda")
    h[:K * W].view(K, W).copy_(torch.from_numpy(b).cuda().expand(K, W))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    peak = {"device": 0}
    yield b, h, peak
    free, total = torch.cuda.mem_get_info()
    peak.pop("host", None)
    print(f"\npast 4 GiB on {torch.cuda.get_device_name()}: {time.perf_counter() - t0:.1f} s, peak device "
          f"memory in use {max(peak['device'], total - free) / 2**30:.1f} GiB (torch's own peak "
          f"{torch.cuda.max_memory_allocated() / 2**30:.1f} GiB)")
    del h
    torch.cuda.empty_cache()


def _note_memory(torch, peak):
    free, total = torch.cuda.mem_get_info()
    peak["device"] = max(peak["device"], total - free)


def _device_i64(torch, ptr, rows, cols):
    """rows x cols int64 view of library-owned device memory (not copied)"""
    class Dev:
        __cuda_array_interface__ = {"shape": (rows, cols), "typestr": "<i8", "data": (ptr, False), "version": 2}
    return torch.as_tensor(Dev(), device="cuda")


def _check_periodic(torch, got, base: np.ndarray, step, what: str):
    """got (K * c rows) == copy j of base + j * step for every copy j, compared on the device"""
    c = base.shape[0]
    assert got.shape[0] == K * c, f"{what}: {got.shape[0]} rows, want {K} x {c}"
    b = torch.from_numpy(base.astype(np.int64)).cuda()
    s = torch.tensor(step, dtype=torch.int64, device="cuda")
    for j0 in range(0, K, 100):  # (in chunks of copies: the expectation is as large as the result)
        j1 = min(K, j0 + 100)
        want = b[None] + torch.arange(j0, j1, device="cuda")[:, None, None] * s
        bad = torch.nonzero((got[j0 * c:j1 * c].view(j1 - j0, c, -1) != want).any(dim=2))
        assert bad.numel() == 0, f"{what}: {bad.shape[0]} rows differ, first (copy, row) {bad[:3].tolist()}"


@pytest.mark.parametrize("flags", FLAG_SETS, ids=lambda f: "+".join(sorted(f)) or "none")
@pytest.mark.parametrize("sf", list(STORES), ids=lambda sf: "".join(map(str, sf)))
def test_whole_call_equals_copy_zero_shifted(torch, store_cache, periodic, sf, flags):
    b, h, peak = periodic
    pats = inputs.case_patterns(dict(patterns="names", store_flags=sf))
    assert b"0" not in pats
    path = store_cache(STORES[sf], pats, sf)
    want = Oracle.from_olm(path).match(b, **flags)
    c0, n = want.size, K * W
    assert c0 > 1000
    base = np.stack([want["offset"], want["len"]], axis=1)
    with Matcher(path) as m:
        cnt, ptr = m.match_device(h.data_ptr(), n, **flags)
        rec = _device_records(torch, ptr, cnt)
        _note_memory(torch, peak)
        _check_periodic(torch, torch.stack([rec[:, 0], rec[:, 1] & 0xFFFFFFFF], dim=1), base, [W, 0], "records")
        assert bool((rec[:, 2] == rec[:, 0] + h.data_ptr()).all())

        # lines: copy j's positions are copy 0's + (j * newlines of B, j * W, j * W)
        pos = torch.zeros((cnt, 3), dtype=torch.int64, device="cuda")
        m.line_positions_device(rec.data_ptr(), cnt, h.data_ptr(), 0, n, pos.data_ptr())
        pos0 = positions(b, want["offset"])
        nl = int((b == 10).sum())
        _check_periodic(torch, pos, pos0, [nl, W, W], "line positions")
        n_lines, lp = m.matching_lines_device(pos.data_ptr(), cnt)
        _note_memory(torch, peak)
        _check_periodic(torch, _device_i64(torch, lp, n_lines, 4), _rle(pos0), [nl, W, W, 0], "matching lines")
        del pos

        # the listing of the last two copies: offsets of 10 digits
        last = rec[(K - 2) * c0:]
        tptr, tlen = m.format_records_device(last.data_ptr(), 2 * c0, h.data_ptr(), 0)
        got = bytes(torch.as_tensor(_DevBytes(tptr, tlen), device="cuda").cpu().numpy())
        bb = b.tobytes()
        text = b"".join(b"%d:%s\n" % (j * W + o, bb[o:o + k].split(b"\0")[0])
                        for j in (K - 2, K - 1) for o, k in zip(want["offset"].tolist(), want["len"].tolist()))
        assert got == text

        # pattern ids: every copy has copy 0's; the counts are K x copy 0's
        m.set_pattern_ids(True)
        cnt2, ptr2 = m.match_device(h.data_ptr(), n, **flags)
        assert cnt2 == cnt
        ids = (_device_i64(torch, ptr2, cnt2, 3)[:, 1] >> 32).view(K, c0)
        torch.cuda.synchronize()  # (read before the next call reuses the records' memory)
        assert bool((ids[0] < m.pattern_count).all())
        bad = torch.nonzero((ids != ids[0]).any(dim=1)).flatten()
        assert bad.numel() == 0, f"ids of copies {bad[:5].tolist()} differ from copy 0"
        counts = torch.zeros(m.pattern_count, dtype=torch.int64, device="cuda")
        assert m.pattern_counts_device(h.data_ptr(), n, counts.data_ptr(), **flags) == cnt
        assert torch.equal(counts, K * torch.bincount(ids[0], minlength=m.pattern_count))
        m.set_pattern_ids(False)
        _note_memory(torch, peak)

        if sf == (0, 0, 0):  # the segmented host path on the host copy of H
            if "host" not in peak:
                peak["host"] = h[:n].cpu().numpy()
            got = m.match_arrays(peak["host"], **flags)
            dev = _as_matches(rec)
            assert got.size == cnt and (got["offset"] == dev["offset"]).all() and (got["len"] == dev["len"]).all()
