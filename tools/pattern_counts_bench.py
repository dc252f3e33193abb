#!/usr/bin/env python3
"""pattern_counts_bench.py -- what counting matches per pattern costs (include/olm_b200.h "pattern counts").

For each workload (bench.py's WORKLOADS, patterns and device-resident haystacks, imported from there):
  device  median olm_cuda_timing_t.total_ms of match_device with ids off, match_device with ids on,
          and count_patterns_device, alternating after warm-up.  On cfg5 and names also the two
          histograms of the counting kernel forced (OLM_COUNT_TABLE=0: warp aggregation and global
          adds; =1: with the per-block shared-memory table), next to the one the library selects.
  host    wall time from pinned host memory of pattern_counts() against match_ids() + np.bincount.
  check   the counts equal a torch.bincount of the ids of the ids-on device records, and the host
          counts equal the device counts.
One JSON line on stdout, with the card's name and power limit read in the same run.

  python tools/pattern_counts_bench.py [--workloads cfg5,names,census-cpw] [--rounds 5] [--warmup 2]
"""
from __future__ import annotations

import argparse
import os
import re
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))

import bench  # noqa: E402  (points fd 1 at stderr; the result line goes out through bench.emit)
from pattern_ids_bench import N_PATTERNS, SIZES, card  # noqa: E402

VARIANTS = ("cfg5", "names")  # where the two histograms are both timed


def matcher(olm: str, dev, table=None):
    """A matcher whose counting histogram is the library's choice, or forced (engine reads it at create)."""
    from omega_match_b200 import Matcher
    if table is None:
        os.environ.pop("OLM_COUNT_TABLE", None)
    else:
        os.environ["OLM_COUNT_TABLE"] = table
    try:
        return Matcher(olm, device=dev.index)
    finally:
        os.environ.pop("OLM_COUNT_TABLE", None)


def run_workload(torch, synth_torch, name: str, tmp: str, args, dev) -> dict:
    from omega_match_b200 import Compiler
    pats, sflags, mflags, hay_kind = bench.workload_patterns(name, N_PATTERNS.get(name, 0))
    n = SIZES[name]
    olm = str(Path(tmp) / f"counts_{name}.olm")
    t0 = time.time()
    Compiler.compile_from_buffer(olm, b"\n".join(pats) + b"\n", *map(bool, sflags))
    gen, _ = bench.device_haystack(torch, synth_torch, hay_kind, pats, 0, n, dev)
    hay = torch.empty(n + 256, dtype=torch.uint8, device=dev)
    hay[:n] = gen
    hay[n:] = 0
    del gen
    torch.cuda.synchronize()
    bench.log(f"[counts] {name}: {len(pats)} patterns, {n} bytes, set up in {time.time() - t0:.1f}s")
    m = matcher(olm, dev)
    P = m.pattern_count
    counts = torch.zeros(P, dtype=torch.int64, device=dev)
    forced = {t: matcher(olm, dev, t) for t in ("0", "1")} if name in VARIANTS else {}

    def match(ids: bool):
        m.set_pattern_ids(ids)
        cnt, ptr = m.match_device(hay.data_ptr(), n, **mflags)
        return cnt, ptr, m.last_timing()["total_ms"]

    def count(mm):
        counts.zero_()
        total = mm.pattern_counts_device(hay.data_ptr(), n, counts.data_ptr(), **mflags)
        return total, mm.last_timing()["total_ms"]

    calls = {"ids_off": lambda: match(False)[2], "ids_on": lambda: match(True)[2], "count": lambda: count(m)[1]}
    for t, mm in forced.items():
        calls[f"count_table{t}"] = lambda mm=mm: count(mm)[1]
    for _ in range(args.warmup):
        for f in calls.values():
            f()
    ms = {k: [] for k in calls}
    for _ in range(args.rounds):
        for k, f in calls.items():
            ms[k].append(f())
    med = {k: float(np.median(v)) for k, v in ms.items()}

    # check: the counts against a bincount of the ids-on records, for every histogram
    cnt_on, ptr, _ = match(True)
    rec = torch.as_tensor(bench.DevArray(ptr, cnt_on), device=dev)
    want = torch.bincount((rec[:, 1] >> 32) & 0xFFFFFFFF, minlength=P)
    del rec
    m.set_pattern_ids(False)
    for mm in [m] + list(forced.values()):
        total, _ = count(mm)
        if total != cnt_on or not bool((counts == want).all()):
            raise SystemExit(f"{name}: the counts differ from a bincount of the ids-on records")
    for mm in forced.values():
        mm.destroy()

    # host path from pinned memory: pattern_counts() against match_ids() + np.bincount
    host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    host.copy_(hay[:n])
    hnp = host.numpy()
    del hay
    torch.cuda.empty_cache()

    def host_counts():
        t = time.perf_counter()
        c = m.pattern_counts(hnp, **mflags)
        return time.perf_counter() - t, c

    def host_ids():
        t = time.perf_counter()
        c = np.bincount(m.match_ids(hnp, **mflags)["pattern_id"], minlength=P)
        return time.perf_counter() - t, c

    host_counts(), host_ids()  # warm-up
    wall = {"pattern_counts": [], "match_ids_bincount": []}
    for _ in range(args.host_rounds):
        t1, c1 = host_counts()
        t2, c2 = host_ids()
        wall["pattern_counts"].append(t1 * 1e3)
        wall["match_ids_bincount"].append(t2 * 1e3)
    if not (np.array_equal(c1, c2.astype(np.uint64)) and np.array_equal(c1, want.cpu().numpy().astype(np.uint64))):
        raise SystemExit(f"{name}: host counts differ")
    selected = "table" if bench_selects_table(cnt_on, P) else "no_table"
    m.destroy()
    del host, hnp
    res = {"bytes": n, "patterns": P, "records": int(cnt_on), "records_per_pattern": round(cnt_on / P, 2),
           "match_flags": sorted(mflags), "selected_histogram": selected}
    for k in calls:
        res[f"ms_{k}"] = round(med[k], 3)
    res["count_over_ids_on"] = round(med["count"] / med["ids_on"], 4)
    for k, v in wall.items():
        res[f"host_ms_{k}"] = round(float(np.median(v)), 1)
    res["device_ms_all"] = {k: [round(x, 3) for x in v] for k, v in ms.items()}
    res["host_ms_all"] = {k: [round(x, 1) for x in v] for k, v in wall.items()}
    res["counts_equal_bincount_of_ids"] = True
    return res


def bench_selects_table(records: int, patterns: int) -> bool:
    """The library's rule (pattern_ids.cu pattern_counts_block_table) with its threshold read from there."""
    src = (ROOT / "omega_match_b200" / "csrc" / "pattern_ids.cu").read_text()
    m = re.search(r"constexpr uint64_t kCountTableMinRepeat = (\d+);", src)
    if not m:
        raise SystemExit("pattern_ids.cu: kCountTableMinRepeat not found")
    return records >= int(m.group(1)) * patterns


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg5,names,census-cpw")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--host-rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import synth_torch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    line = {"tool": "pattern_counts_bench", "gpu": card(0),
            "unit_ms": "device ms per call (olm_cuda_timing_t.total_ms); host: wall ms per call from pinned memory",
            "workloads": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for w in args.workloads.split(","):
            res = run_workload(torch, synth_torch, w, tmp, args, dev)
            line["workloads"][w] = res
            bench.log(f"[counts] {w}: {res}")
    bench.emit(line)


if __name__ == "__main__":
    main()
